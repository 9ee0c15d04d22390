#!/usr/bin/env python
"""bench.py -- snapshot-stream GiB/s of the peer-bootstrap hot path on B200.

Headline workload = BASELINE.json configs[2], the config its `metric` ("Fletcher-4+LZ4") is quoted
on: a 64 GiB (logical) ZFS-send stream of LZ4-compressed 128 KiB records, mode RECOMPRESS
(decode -> verify every stream checksum -> re-encode with the declared ZFS encoder -> re-stamp).
One "step" = one full pass of the stage over that stream.  The metric counts INPUT STREAM bytes
(SURVEY.md 8d: wire-format bytes, headers + compressed payloads, BEGIN...END) per second.

  value     whole-job GiB/s with the stream resident in HBM (mtz_dev_submit / mtz_dev_finish[_exchange],
            CUDA events on the launching stream, max over ranks)
  e2e       the same through the host-facing C-ABI call a caller makes (mtz_process_host, pinned host
            buffers in and out, H2D + D2H inside the timed region).  With N GPUs it is ONE process
            driving the device group mtz_config.devices[0..N) -- what a Node backupserver would do.
  e2e_stream_api   the ring API the N-API Transform binds (acquire/commit, write, peek/consume)
  roofline  K3 (LZ4 encode, the dominant kernel) algorithmic HBM bytes / its CUDA-event time
  cpu_baseline / --impl reference
            the oracle port of the same arithmetic on all host threads (oracle/mt.c), on a bounded
            sample of the same workload.  Reported, not the target.

N > 1 (torchrun, one rank per GPU): STRONG scaling of the same 64 GiB stream, partitioned by record
index into N contiguous shards; the only data-path exchange is the library-owned NCCL all-gather of
the 40-byte shard aggregate plus the 32-byte output checksum hopping rank to rank
(mtz_dev_finish_exchange).  Rank 0 then measures, in one process over all N GPUs, `e2e` and the
fan-out of the processed stream to P attached peers (BASELINE configs[3]/[4]).

`--dump-outputs DIR` writes, after the timed steps, what the last timed step returned as DIR/<name>.npy
(float32 / float64, u64 values as exact (hi32, lo32) pairs): per chunk j the output stream's size
(chunkj_output_bytes), the running checksums the finish call returned (chunkj_carry, chunkj_carry_out)
and 128 / (number of chunks) windows of 64 KiB of the output stream at seeded offsets
(chunkj_output_sample, chunkj_output_sample_offsets), plus the END checksum (end_checksum); with
`--workload verify` the step's size, carries and END checksum; with `--impl reference` what the oracle
returned for its bounded sample, under the same names without the chunk prefix.  The inputs
are seeded, so two builds run with the same arguments can be compared array for array.

`--workload verify` keeps round 1's headline (configs[1]: 16 GiB uncompressed, Fletcher-4 only) as a
selectable workload; the default run reports it as `workloads.verify`.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GIB = float(1 << 30)
RECSIZE = 131072
REC_BYTES = 312 + RECSIZE


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="recompress", choices=["recompress", "verify"])
    ap.add_argument("--gib", type=float, default=0.0,
                    help="workload size: logical GiB of the whole job (recompress, default 64) / "
                         "stream GiB per GPU (verify, default 16)")
    ap.add_argument("--ref-gib", type=float, default=8.0,
                    help="CPU arms: GiB (logical for recompress) of the bounded sample each step processes")
    ap.add_argument("--verify-gib", type=float, default=16.0, help="side workload (N=1), 0 = skip")
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-reencode", action="store_true", help="skip the certificate-off resident leg (N=1)")
    ap.add_argument("--recsize", type=int, default=131072, help="DRR_WRITE logical size (dataset recordsize)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy "
                         "(see the module docstring), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for (ts, r) in self.rows if t0 is None or (t0 - 0.02 <= ts <= t1 + 0.05)]
        scope = "timed region"
        if len(rows) < 2:             # region shorter than the sampler's period: use the whole
            rows = [r for (ts, r) in self.rows]      # loaded window (warm-up + timed steps)
            scope = "warm-up + timed region"
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except ValueError:
                continue
            for nm, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None,
                "samples": len(sm), "scope": scope, "reasons": sorted(reasons)}


SIMD_NAME = {0: "scalar", 4: "avx2 (4 lanes, as zfs_fletcher_avx2)", 8: "avx512f (8 lanes, as zfs_fletcher_avx512)"}


def cpu_quota():
    """cgroup CPU quota in cores (None = unlimited): shared GPU boxes often cap it"""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        return None if q == "max" else round(float(q) / float(per), 2)
    except Exception:
        return None


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def load_peaks():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (a STREAM copy, read+write)"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


# ------------------------------------------------------------------ CPU legs (oracle port) --
def cpu_verify_baseline(O, stream, nthreads):
    """cpu_baseline object of the VERIFY workload: the oracle port over `stream` on `nthreads`
    threads, plus the one-thread figure -- the shape a real `zfs send` / `zfs recv` stream checksum
    has."""
    rc, secs, cst = O.mt_verify(stream, nthreads)
    assert rc == 0, rc
    rc, secs, cst = O.mt_verify(stream, nthreads)          # second pass: buffers warm
    assert rc == 0, rc
    rc, secs1, _ = O.mt_verify(stream, 1)
    assert rc == 0, rc
    lanes = O.simd_lanes()
    flavour = SIMD_NAME.get(lanes, "scalar")
    return {"value": round(stream.size / GIB / secs, 3), "unit": "GiB/s", "cores": nthreads,
            "cgroup_cpu_quota": cpu_quota(), "kind": "port", "fletcher4": flavour,
            "single_thread_value": round(stream.size / GIB / secs1, 3),
            "sample": "the whole %.2f GiB stream, second of two passes: record-parallel %s fletcher_4 "
                      "(oracle/mt.c), %d threads; single_thread_value = one thread, the shape of a real "
                      "`zfs send`/`zfs recv` stream checksum" % (stream.size / GIB, flavour, nthreads)}


def cpu_recompress(O, src, out, nthreads):
    """one oracle RECOMPRESS pass (record-parallel LZ4 decode + encode, vector Fletcher-4, sequential
    stamp) -> (output bytes, seconds)"""
    import ctypes as C
    L = O.lib()
    n = C.c_size_t(0); st = O.StreamStats(); secs = C.c_double(0)
    rc = L.orc_mt_recompress(src.ctypes.data, src.size, out.ctypes.data, out.size, C.byref(n),
                             nthreads, C.byref(secs), C.byref(st))
    assert rc == 0, rc
    return n.value, secs.value


def make_lz4_stream(O, logical_gib, nthreads, pinned=True):
    """The configs[2] input: `logical_gib` of pg-page 128 KiB records (SURVEY 8d payload model), each
    stored as the declared encoder's ZFS-LZ4 frame, checksums stamped -- i.e. what `zfs send -c` of
    an lz4 dataset carries.  Returns (stream array, logical bytes, holder to free)."""
    import numpy as np
    nwrites = max(1, int(logical_gib * GIB) // REC_BYTES)
    raw = O.synth_stream(nwrites, RECSIZE, O.PAYLOAD_PGPAGE, nthreads=nthreads)
    logical = float(raw.size)
    cbuf = np.empty(raw.size + (1 << 20), dtype=np.uint8)
    n, _ = cpu_recompress(O, raw, cbuf, nthreads)          # raw -> oracle-encoded LZ4 stream
    del raw
    O.lib().orc_mt_release()                               # its scratch is as large as `raw` was
    if not pinned:
        return cbuf[:n].copy(), logical, None
    from manatee_b200 import PinnedBuffer
    pin = PinnedBuffer(n)
    pin.array[:] = cbuf[:n]
    return pin.array, logical, pin


def recompress_config(total_logical_gib, stream_bytes=None, records=None, ratio=None):
    """`config` of the RECOMPRESS workload -- the SAME object on both arms."""
    return {"workload": "recompress: %.0f GiB logical ZFS-send stream of LZ4-compressed 128 KiB records, "
                        "decode + Fletcher-4 verify + re-encode + re-stamp (BASELINE configs[2])" % total_logical_gib,
            "recordsize": RECSIZE, "payload": "pg-page model, Zipf dictionary seed 0x5047 (LZ4 ratio ~2.5)",
            "metric_bytes": "input stream bytes (312 B headers + compressed payloads, BEGIN..END)"}


def verify_config(gib_per_gpu):
    return {"workload": "verify: %.0f GiB/GPU uncompressed ZFS-send stream, Fletcher-4 (BASELINE configs[1])" % gib_per_gpu,
            "recordsize": RECSIZE, "payload": "PCG32 seed 0x4D414E41 (incompressible)",
            "metric_bytes": "input stream bytes"}


# ------------------------------------------------------------------------------ output dump --
DUMP_WINDOW = 65536          # bytes per sampled window of an output stream
DUMP_SAMPLE_BYTES = 8 << 20  # sampled output bytes over all chunks: 32 MiB as float32


def u64_words(vals):
    """u64 values as float64 (hi32, lo32) pairs: exact, unlike a u64 -> float64 cast"""
    import numpy as np
    v = np.asarray(vals, dtype=np.uint64).reshape(-1)
    return np.stack([v >> np.uint64(32), v & np.uint64(0xffffffff)], axis=1).astype(np.float64)


def output_sample(d_out, out_bytes, in_bytes, seed, windows):
    """`windows` windows of DUMP_WINDOW bytes of the device output stream d_out[:out_bytes] at
    offsets drawn with `seed` over the INPUT size, which is identical between builds -> (bytes as
    float32, -1 past the end of the output; window offsets as float64)"""
    import numpy as np
    import torch
    rng = np.random.default_rng(seed)
    offs = np.sort(rng.integers(0, max(1, in_bytes - DUMP_WINDOW + 1), size=windows))
    idx = (torch.from_numpy(offs).to(d_out.device)[:, None] +
           torch.arange(DUMP_WINDOW, device=d_out.device)[None, :]).reshape(-1)
    vals = d_out[idx.clamp(max=max(0, out_bytes - 1))].float()
    vals[idx >= out_bytes] = -1.0
    return vals.cpu().numpy(), offs.astype(np.float64)


def dump_outputs(dirname, arrays):
    """DIR/<name>.npy for every array, float32 / float64 only"""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(dirname, name + ".npy"), a)


# ----------------------------------------------------------------------------- reference arm --
def run_reference(args):
    """CPU arm: the oracle port of the path's arithmetic on all host threads, each step a bounded
    sample of the arm's workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import numpy as np
    import oracle as O
    O.build()
    nthreads = host_threads()
    note = ("reference = Node identity pipe + in-kernel ZFS arithmetic (`zfs send`/`zfs recv`, "
            "lib/backupSender.js:177, lib/zfsClient.js:793); node/zfs are not installable here, so the "
            "oracle port of that arithmetic is timed (kind=port), record-parallel over every host thread "
            "-- more parallelism than the reference's single `zfs send` thread has")
    if args.workload == "verify":
        gib = args.gib or 16.0
        nwrites = max(1, int(min(args.ref_gib * 2, gib) * GIB) // REC_BYTES)
        s = O.synth_stream(nwrites, RECSIZE, O.PAYLOAD_PCG, nthreads=nthreads)
        for _ in range(max(1, min(args.warmup, 2))):
            assert O.mt_verify(s, nthreads)[0] == 0
        t = []
        for _ in range(args.steps):
            rc, secs, st = O.mt_verify(s, nthreads)
            assert rc == 0
            t.append(secs)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"end_checksum": u64_words(st.end_cksum.tuple())})
        ms = 1e3 * sum(t) / len(t)
        val = s.size / GIB / (ms / 1e3)
        cfg = verify_config(gib)
        sample = ("%.2f GiB of the stream per step: record-parallel %s fletcher_4 + sequential combine "
                  "(oracle/mt.c)" % (s.size / GIB, SIMD_NAME.get(O.simd_lanes(), "scalar")))
        dtype = "u32->u64 (mod 2^64)"
    else:
        gib = args.gib or 64.0
        src, logical, _ = make_lz4_stream(O, min(args.ref_gib, gib), nthreads, pinned=False)
        out = np.empty(src.size + (1 << 20), dtype=np.uint8)
        for _ in range(max(1, min(args.warmup, 2))):
            n, _s = cpu_recompress(O, src, out, nthreads)
        assert n == src.size and np.array_equal(out[:n], src), "oracle RECOMPRESS is not idempotent"
        t = []
        for _ in range(args.steps):
            n, secs = cpu_recompress(O, src, out, nthreads)
            t.append(secs)
        if args.dump_outputs:
            import torch
            smp, offs = output_sample(torch.from_numpy(out), n, src.size, seed=0x4d545a,
                                      windows=DUMP_SAMPLE_BYTES // DUMP_WINDOW)
            dump_outputs(args.dump_outputs, {"output_sample": smp, "output_sample_offsets": offs,
                                             "output_bytes": np.array([n], dtype=np.float64)})
        ms = 1e3 * sum(t) / len(t)
        val = src.size / GIB / (ms / 1e3)
        cfg = recompress_config(gib)
        sample = ("%.2f GiB logical (%.2f GiB of input stream) of the workload per step: record-parallel "
                  "oracle LZ4 decode + encode + vector Fletcher-4, sequential stamp (oracle/mt.c); "
                  "logical %.2f GiB/s" % (logical / GIB, src.size / GIB, logical / GIB / (ms / 1e3)))
        dtype = "u8 / u32->u64 (mod 2^64)"
    line = {
        "impl": "reference", "metric": "snapshot_stream_gibs", "value": round(val, 3),
        "unit": "GiB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms, 3), "higher_is_better": True,
        "scaling": "strong" if args.workload == "recompress" else "weak",
        "vs_baseline": None, "dtype": dtype, "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": round(val, 3), "unit": "GiB/s", "cores": nthreads,
                         "cgroup_cpu_quota": cpu_quota(), "kind": "port", "sample": sample},
        "e2e": {"value": round(val, 3), "unit": "GiB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "note": note,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------- ring API helpers --
_PUMP = None


def ring_pump():
    """tools/libringpump.so: native producers for the ring API (bench infrastructure, built by
    __graft_entry__.build(); rebuilt here if it did not travel)."""
    global _PUMP
    if _PUMP is None:
        import ctypes as C
        so = os.path.join(ROOT, "tools", "libringpump.so")
        if not os.path.exists(so):
            subprocess.check_call(["gcc", "-O2", "-shared", "-fPIC", "-pthread", "-o", so,
                                   os.path.join(ROOT, "tools", "ringpump.c")])
        P = C.CDLL(so)
        P.pump_memcpy.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int]
        P.pump_memcpy.restype = C.c_int32
        P.pump_pipe.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t]
        P.pump_pipe.restype = C.c_int32
        P.pump_selfcopy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_int]
        P.pump_selfcopy.restype = C.c_int32
        _PUMP = P
    return _PUMP


def pump_threads():
    """memcpy threads of the native producer: half of what the process may use (the cgroup quota
    counts), so that the library's engine thread and the CUDA callback thread are not starved"""
    q = cpu_quota()
    n = min(host_threads(), int(q)) if q else host_threads()
    return max(2, min(12, (3 * n) // 4))


def host_memcpy_ceiling(src, nthreads, chunk=64 << 20):
    """GiB/s of the producer alone: the pump's parallel memcpys from `src` into one pinned 64 MiB
    slice, no library behind it -- what an acquire/commit leg cannot exceed on this host."""
    from manatee_b200 import PinnedBuffer
    pin = PinnedBuffer(chunk)
    n = min(src.size, 8 << 30)
    P = ring_pump()
    t0 = time.perf_counter()
    P.pump_selfcopy(pin.array.ctypes.data, src.ctypes.data, n, chunk, nthreads)
    dt = time.perf_counter() - t0
    pin.free()
    return round(n / GIB / dt, 3)


def ring_run(g, src, peers=(0,), producer="write", nthreads=4, chunk=64 << 20, limit_s=240.0):
    """Drive the streaming API: one producer feeding `src` (numpy u8), one zero-copy consumer thread
    per peer (mtz_out_peek_peer / mtz_out_consume_peer).  producer = "write" (mtz_write: one thread,
    one memcpy into the pinned ring), "acquire" (mtz_ring_acquire / commit, the slice filled by
    `nthreads` parallel memcpys, native: tools/ringpump.c) or "pipe" (a pipe(2) read(2) straight into
    the acquired slice -- the shape of zfsSend.stdout).  Returns (seconds, ok, detail).  A leg that has not
    finished after `limit_s` is cancelled (mtz_cancel) and reported as failed: a stuck leg must not cost
    the JSON line."""
    import ctypes as C
    from manatee_b200 import _native as N
    L = N.lib()
    errs, got = [], {}

    def consumer(p):
        try:
            ptr, n, tot = C.c_void_p(), C.c_size_t(), 0
            while True:
                rc = L.mtz_out_peek_peer(g._h, p, C.byref(ptr), C.byref(n))
                if rc == N.OK:
                    tot += n.value
                    L.mtz_out_consume_peer(g._h, p, n.value)
                elif rc == N.EOF:
                    break
                elif rc == N.EAGAIN:
                    time.sleep(0.0002)
                else:
                    errs.append("peer %d: rc %d" % (p, rc))
                    break
            got[p] = tot
        except Exception as e:              # noqa: BLE001
            errs.append(repr(e))

    def produce():
        try:
            if producer == "write":
                for o in range(0, src.size, chunk):
                    g.write(src[o:o + chunk])
            else:
                P = ring_pump()
                acq = C.cast(L.mtz_ring_acquire, C.c_void_p)
                com = C.cast(L.mtz_ring_commit, C.c_void_p)
                if producer == "acquire":
                    rc = P.pump_memcpy(acq, com, g._h, src.ctypes.data, src.size, chunk, nthreads)
                else:
                    rc = P.pump_pipe(acq, com, g._h, src.ctypes.data, src.size, chunk)
                if rc != 0:
                    raise RuntimeError("ring pump rc %d: %s" % (rc, (L.mtz_last_error(g._h) or b"").decode()))
            g.flush()
        except Exception as e:              # noqa: BLE001
            errs.append(repr(e))
            g.cancel()

    # the handle builds its engine lazily (pinned rings of a GiB each, GPU slots, the NCCL group for
    # a fan-out): an empty acquire/commit does that BEFORE the clock starts -- a long-lived daemon
    # pays it once per restore, not per GiB
    _p, _n = C.c_void_p(), C.c_size_t()
    rc0 = L.mtz_ring_acquire(g._h, 1, C.byref(_p), C.byref(_n))
    if rc0 == N.OK:
        L.mtz_ring_commit(g._h, 0)
    ts = [threading.Thread(target=consumer, args=(p,)) for p in peers]
    t0 = time.perf_counter()
    tp = threading.Thread(target=produce)
    tp.start()
    for t in ts:
        t.start()
    deadline = time.time() + limit_s
    for t in [tp] + ts:
        t.join(max(0.0, deadline - time.time()))
    if any(t.is_alive() for t in [tp] + ts):
        errs.append("leg not finished after %.0f s: cancelled" % limit_s)
        g.cancel()
        for t in [tp] + ts:
            t.join(30.0)
    dt = time.perf_counter() - t0
    return dt, (not errs), {"errors": errs[:3], "delivered": got}


# -------------------------------------------------------------------------------- our arm --
def run_verify_resident(args, O, local, steps, warm, peak):
    """configs[1] on one GPU: 16 GiB uncompressed stream resident in HBM; GPU parse + K1 + scan per
    step (round 1's headline, kept as a workload)."""
    import numpy as np
    import torch
    from manatee_b200 import GpuSnapshotStage, PinnedBuffer, index_host
    gib = args.verify_gib if args.workload != "verify" else (args.gib or 16.0)
    nthreads = host_threads()
    nwrites = max(1, int(gib * GIB) // REC_BYTES)
    nbytes = O.lib().orc_synth_stream_size(nwrites, RECSIZE)
    pin = PinnedBuffer(nbytes)
    s = O.synth_stream(nwrites, RECSIZE, O.PAYLOAD_PCG, nthreads=nthreads, out=pin.array)
    recs, used = index_host(s)
    assert used == s.size
    d_stream = torch.empty(s.size + 512, dtype=torch.uint8, device="cuda")
    d_stream[:s.size].copy_(torch.from_numpy(s))
    d_recs = torch.empty((len(recs) + 16) * 32, dtype=torch.uint8, device="cuda")
    st = torch.cuda.Stream()
    res = {}
    with GpuSnapshotStage("verify", device=local) as g:
        def step():
            n_idx, used_idx = g.dev_index(d_stream.data_ptr(), s.size, d_recs.data_ptr(), len(recs) + 16,
                                          cuda_stream=st.cuda_stream)
            assert n_idx == len(recs) and used_idx == s.size
            g.dev_submit(d_stream.data_ptr(), s.size, d_recs.data_ptr(), n_idx, cuda_stream=st.cuda_stream)
            return g.dev_finish(carry_in=(0, 0, 0, 0))
        for _ in range(warm):
            step()
        s0 = g.stats()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(st)
        for _ in range(steps):
            fin = step()
        e1.record(st)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        s1 = g.stats()
        k1_ms = (s1["k1_ms"] - s0["k1_ms"]) / max(1, s1["k1_launches"] - s0["k1_launches"])
        end_ck = g.end_checksum()
        if args.dump_outputs and args.workload == "verify":
            # VERIFY hands the input on unchanged: what a step returns is its verdict
            dump_outputs(args.dump_outputs, {"output_bytes": np.array([fin[0]], dtype=np.float64),
                                             "carry": u64_words(fin[1]), "carry_out": u64_words(fin[2]),
                                             "end_checksum": u64_words(end_ck)})
        res.update({"value": round(s.size / GIB / (ms / 1e3), 3), "unit": "GiB/s", "ms_per_step": round(ms, 4),
                    "steps": steps, "gpu_launches": int((s1["kernel_launches"] - s0["kernel_launches"]) // steps),
                    "config": verify_config(gib),
                    "roofline": {"bound": "hbm", "kernel": "k1_record_sums",
                                 "achieved": round(s.size / (k1_ms / 1e3) / 1e9, 1), "peak": peak, "unit": "GB/s",
                                 "frac": round(s.size / (k1_ms / 1e3) / 1e9 / peak, 4), "traffic": None,
                                 "algorithmic_bytes_per_launch": float(s.size), "k1_ms": round(k1_ms, 4),
                                 "note": "K1 only reads; the peak is a copy (read+write), so ~1.0 is the roof"}})
    del d_stream, d_recs
    torch.cuda.empty_cache()
    if not args.no_e2e:
        with GpuSnapshotStage("verify", device=local, batch_bytes=64 << 20, n_slots=4) as ge:
            ge.process_host(s)
            t0 = time.perf_counter()
            k = max(1, min(steps, args.e2e_steps))
            for _ in range(k):
                ge.process_host(s)
            dt = (time.perf_counter() - t0) / k
        res["e2e"] = {"value": round(s.size / GIB / dt, 3), "unit": "GiB/s",
                      "h2d_bytes_per_step": int(s.size + len(recs) * 32),
                      "d2h_bytes_per_step": int(((s.size + (64 << 20) - 1) // (64 << 20)) * 120),
                      "call": "mtz_process_host, pinned host stream in, verdict out (output == input)"}
        # the ring API at link rate: acquire/commit, the slice filled by parallel memcpys
        with GpuSnapshotStage("verify", device=local, ring_bytes=1 << 30, batch_bytes=64 << 20, n_slots=4) as gr:
            nt = pump_threads()
            dt, ok, det = ring_run(gr, s, producer="acquire", nthreads=nt)
            res["ring_acquire_commit"] = {"value": round(s.size / GIB / dt, 3), "unit": "GiB/s", "ok": bool(
                ok and det["delivered"].get(0) == s.size and gr.end_checksum() == end_ck),
                "producer_threads": nt, "host_memcpy_ceiling_gibs": host_memcpy_ceiling(s, nt),
                "call": "mtz_ring_acquire/commit (slices filled by parallel host memcpys) -> engine -> "
                        "mtz_out_peek/consume in place (zero copy)"}
    if not args.no_cpu:
        rc, secs, cst = O.mt_verify(s, nthreads)
        assert rc == 0 and cst.end_cksum.tuple() == end_ck, "GPU END checksum differs from the oracle's"
        k = int(np.searchsorted(recs["off"], min(s.size, int(4 * GIB)), side="right")) - 1
        cut = s.size if k + 1 >= len(recs) else int(recs["off"][max(1, k)])      # whole records only
        res["cpu_baseline"] = cpu_verify_baseline(O, s[:cut], nthreads)
    res["end_checksum"] = ["%016x" % x for x in (end_ck or ())]
    pin.free()
    return res


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import oracle as O                      # generator, parity checks and the cpu_baseline leg only
    from manatee_b200 import GpuSnapshotStage, PinnedBuffer, comm_unique_id, index_host
    from manatee_b200 import _native as N

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("--gpus %d needs torchrun with one rank per GPU" % args.gpus)
    torch.cuda.set_device(local)
    gl = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        gl = dist.new_group(backend="gloo")          # CPU-side waits must not spin a kernel on the GPUs
    O.build()
    nthreads = host_threads()
    peak, peak_src = load_peaks()

    if args.workload == "verify":
        if world > 1:
            raise SystemExit("--workload verify is the single-GPU configs[1] measurement; the multi-GPU "
                             "line is the recompress workload")
        clocks = ClockSampler(local); clocks.start()
        t0 = time.time()
        r = run_verify_resident(args, O, local, args.steps, args.warmup, peak)
        clk = clocks.stop(t0, time.time())
        line = {"metric": "snapshot_stream_gibs", "value": r["value"], "unit": "GiB/s", "n_gpus": 1,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u32->u64 (mod 2^64)", "data": "synthetic", "config": r["config"],
                "e2e": r.get("e2e"), "gpu_launches": r["gpu_launches"], "roofline": r["roofline"],
                "cpu_baseline": r.get("cpu_baseline"), "e2e_stream_api": r.get("ring_acquire_commit"),
                "clocks": clk, "end_checksum": r["end_checksum"]}
        print(json.dumps(line), flush=True)
        return 0

    # ------------------------------------------------------------------ the stream (rank 0 makes it)
    total_gib = args.gib or 64.0
    shm = "/dev/shm/mtz_bench_%s.bin" % os.environ.get("MASTER_PORT", str(os.getpid()))
    src = pin_in = None
    meta = [None]
    if rank == 0:
        src, logical, pin_in = make_lz4_stream(O, total_gib, nthreads)
        if world > 1:
            with open(shm, "wb") as f:
                f.write(memoryview(src))
        meta = [{"bytes": int(src.size), "logical": float(logical)}]
    if world > 1:
        dist.broadcast_object_list(meta, src=0, group=gl)
        whole = src if rank == 0 else np.memmap(shm, dtype=np.uint8, mode="r", shape=(meta[0]["bytes"],))
    else:
        whole = src
    logical = meta[0]["logical"]
    total_bytes = float(meta[0]["bytes"])
    recs_all, used = index_host(whole)
    assert used == whole.size
    # record-index partition.  N = 1: the whole stream.  N > 1: the stream is cut into C = 4 N chunks
    # of whole records and rank r takes chunks r, r + N, r + 2N, ... -- round-robin, so that the one
    # serial piece of work (the stamp chain, which needs the previous chunk's output checksum) of one
    # rank's chunk runs under the LZ4 kernels of the other ranks' chunks.  With one contiguous shard
    # per rank every chain would queue up behind ALL the LZ4 work.
    nrec_all = len(recs_all)
    CH = 1 if world == 1 else 4
    C_ALL = CH * world
    bounds = [(j * nrec_all) // C_ALL for j in range(C_ALL + 1)]
    nwrites_total = int((recs_all["type"] == 3).sum())
    chunks = []
    for k in range(CH):
        j = k * world + rank
        r0, r1 = bounds[j], bounds[j + 1]
        b0 = int(recs_all["off"][r0])
        b1 = int(recs_all["off"][r1]) if r1 < nrec_all else int(whole.size)
        recs = recs_all[r0:r1].copy()
        recs["off"] -= b0
        d_in = torch.empty(b1 - b0 + 512, dtype=torch.uint8, device="cuda")
        d_in[:b1 - b0].copy_(torch.from_numpy(np.ascontiguousarray(whole[b0:b1])))
        worst = int((np.maximum(recs["lsize"].astype(np.int64), recs["payload"].astype(np.int64)) + 312).sum()) + (1 << 20)
        chunks.append({"j": j, "bytes": b1 - b0, "nrec": len(recs), "d_in": d_in,
                       "d_recs": torch.from_numpy(recs.view(np.uint8).copy()).cuda(),
                       "d_out": torch.empty(worst, dtype=torch.uint8, device="cuda"),
                       "flags": (N.XCHG_FIRST if j == 0 else 0) | (N.XCHG_LAST if j == C_ALL - 1 else 0)})
    if rank != 0:
        del whole
    torch.cuda.synchronize()

    # ------------------------------------------------------------------ resident timing: `value`
    # two handles and two streams alternate over a rank's chunks: the kernels of chunk k+1 are
    # already running when the exchange of chunk k waits for its turn in the chain
    hs = [GpuSnapshotStage("recompress", device=local, flags=N.FLAG_DEFER_VERIFY if world > 1 else 0)
          for _ in range(1 if world == 1 else 2)]
    sts = [torch.cuda.Stream() for _ in hs]
    if world > 1:
        uid = [comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0, group=gl)
        hs[0].comm_init(uid[0], rank, world)        # the library owns the communicator of the exchange
        hs[1].comm_share(hs[0])
    acc = {"k3_ms": 0.0, "codec_ms": 0.0, "k3_launches": 0.0, "kernel_launches": 0.0,
           "lz4_certified": 0.0, "lz4_encoded": 0.0}
    end_ck = [None]
    finished = [None] * CH                 # (out_bytes, carry, carry_out) of each chunk, last step

    def submit(k):
        c, g, st_ = chunks[k], hs[k % len(hs)], sts[k % len(hs)]
        g.dev_reset()
        g.dev_submit(c["d_in"].data_ptr(), c["bytes"], c["d_recs"].data_ptr(), c["nrec"], c["d_out"].data_ptr(),
                     c["d_out"].numel(), cuda_stream=st_.cuda_stream)

    def step():
        for key in acc:
            acc[key] = 0.0
        base, obs = (0, 0, 0, 0), []
        for k in range(min(len(hs), CH)):
            submit(k)
        for k in range(CH):
            g = hs[k % len(hs)]
            if world == 1:
                fin = g.dev_finish()
            else:
                fin = g.dev_finish_exchange(round_base=base, flags=chunks[k]["flags"])
                base = fin[3]
            finished[k] = fin[:3]
            ob = fin[0]
            obs.append(ob)
            s_ = g.stats()                     # dev_reset() zeroes the counters per chunk
            for key in acc:
                acc[key] += float(s_[key])
            ck = g.end_checksum()
            if ck is not None:
                end_ck[0] = ck
            if k + len(hs) < CH:
                submit(k + len(hs))
        return obs

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    obs = []
    for _ in range(max(1, args.warmup)):
        obs = step()
    # size-independent parity at full size: the input was produced by the declared encoder, so
    # RECOMPRESS must reproduce every chunk bit for bit (idempotence), re-stamped checksums included
    ok_all = all(ob == c["bytes"] and bool(torch.equal(c["d_out"][:ob], c["d_in"][:c["bytes"]]))
                 for ob, c in zip(obs, chunks))
    same = torch.tensor([1 if ok_all else 0], device="cuda")
    if world > 1:
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        dist.barrier()
    same = bool(int(same.item()))
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t_wall0 = time.time()
    e0.record(sts[0])
    for _ in range(args.steps):
        step()
    e1.record(sts[(CH - 1) % len(hs)])          # the stream of the last chunk; every finish has synchronised
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    ksum = torch.tensor([acc["k3_ms"], acc["codec_ms"], acc["k3_launches"], acc["kernel_launches"],
                         acc["lz4_certified"], acc["lz4_encoded"]],
                        dtype=torch.float64, device="cuda")       # the last step alone
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(ksum, op=dist.ReduceOp.SUM)
    clk = clocks.stop(t_wall0, time.time()) if rank == 0 else None
    ms_step = float(t.item()) / args.steps
    value = total_bytes / GIB / (ms_step / 1e3)
    k3_ms, codec_ms, k3_launches, launches, n_cert, n_enc = [float(x) for x in ksum.tolist()]
    end_ck = end_ck[0]
    if args.dump_outputs:
        # the last timed step's output stream of every chunk this rank finished (N = 1: the whole
        # stream), sampled, and the checksums and sizes the finish calls returned
        arrays = {}
        for c, (ob, carry, carry_out) in zip(chunks, finished):
            tag = "chunk%d_" % c["j"]
            arrays[tag + "output_sample"], arrays[tag + "output_sample_offsets"] = output_sample(
                c["d_out"], ob, c["bytes"], seed=0x4d545a + c["j"],
                windows=max(1, DUMP_SAMPLE_BYTES // DUMP_WINDOW // C_ALL))
            arrays[tag + "output_bytes"] = np.array([ob], dtype=np.float64)
            arrays[tag + "carry"], arrays[tag + "carry_out"] = u64_words(carry), u64_words(carry_out)
        if end_ck is not None:
            arrays["end_checksum"] = u64_words(end_ck)
        dump_outputs(args.dump_outputs, arrays)
    # the same resident step with the certificate switched off (MTZ_FLAG_REENCODE_ALL): every record
    # goes through the serial matcher -- what RECOMPRESS costs on a stream made by ANOTHER encoder
    reenc = None
    if world == 1 and not args.no_reencode:
        try:
            with GpuSnapshotStage("recompress", device=local, flags=N.FLAG_REENCODE_ALL) as g2:
                c = chunks[0]
                def one():
                    g2.dev_reset()
                    g2.dev_submit(c["d_in"].data_ptr(), c["bytes"], c["d_recs"].data_ptr(), c["nrec"],
                                  c["d_out"].data_ptr(), c["d_out"].numel(), cuda_stream=sts[0].cuda_stream)
                    return g2.dev_finish()[0]
                ob2 = one()
                ok2 = (ob2 == c["bytes"] and bool(torch.equal(c["d_out"][:ob2], c["d_in"][:c["bytes"]])))
                r0 = torch.cuda.Event(enable_timing=True); r1 = torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize(); r0.record(sts[0])
                kk = max(1, min(3, args.steps))
                for _ in range(kk):
                    one()
                r1.record(sts[0]); torch.cuda.synchronize()
                ms2 = r0.elapsed_time(r1) / kk
                s2 = g2.stats()
            reenc = {"value": round(total_bytes / GIB / (ms2 / 1e3), 3), "unit": "GiB/s",
                     "logical_gibs": round(logical / GIB / (ms2 / 1e3), 3), "ms_per_step": round(ms2, 3),
                     "steps": kk, "k3_ms_per_step": round(float(s2["k3_ms"]), 3),
                     "certified_records": int(s2["lz4_certified"]), "output_equals_input": bool(ok2),
                     "what": "MTZ_FLAG_REENCODE_ALL: the certificate off, every record decoded and re-encoded by "
                             "the serial matcher (k3_lz4_encode) -- round 1/2's RECOMPRESS, and what a stream made "
                             "by a different encoder costs"}
        except Exception as e:                  # noqa: BLE001 -- never costs the headline line
            reenc = {"error": repr(e)}
    for g in hs[::-1]:
        g.close()
    del chunks
    torch.cuda.empty_cache()

    # everything below is rank 0 alone (ONE process over all N GPUs); the others wait on the CPU
    e2e = ring = fan = cpu = side = None
    failed = []
    if rank == 0:
        devices = list(range(world)) if world > 1 else None
        nrec = len(recs_all)
        if not args.no_e2e:
            pin_out = PinnedBuffer(int(total_bytes) + (64 << 20))
            with GpuSnapshotStage("recompress", device=local, devices=devices, n_slots=4) as ge:
                n_out = ge.process_host(src, pin_out.array)
                ok = (n_out == src.size and ge.end_checksum() is not None)
                for o in (0, (src.size // 2) & ~4095, max(0, src.size - (64 << 20))):
                    ok = ok and np.array_equal(pin_out.array[o:o + (64 << 20)][:n_out - o], src[o:o + (64 << 20)])
                if not ok:
                    failed.append("e2e output differs from the oracle-encoded input")
                k = max(1, min(args.steps, args.e2e_steps))
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(k):
                    n_out = ge.process_host(src, pin_out.array)
                dt = (time.perf_counter() - t0) / k
            # the same call with the kernels removed: H2D + D2H of every byte through the same
            # pinned buffers, slots and device group -- the host/PCIe ceiling of this box for e2e
            with GpuSnapshotStage("passthrough", device=local, devices=devices, n_slots=4) as gp:
                gp.process_host(src, pin_out.array)
                t0 = time.perf_counter()
                gp.process_host(src, pin_out.array)
                copy_only = round(total_bytes / GIB / (time.perf_counter() - t0), 3)
            e2e = {"value": round(total_bytes / GIB / dt, 3), "unit": "GiB/s",
                   "logical_gibs": round(logical / GIB / dt, 3), "steps": k,
                   "h2d_bytes_per_step": int(total_bytes + nrec * 32), "d2h_bytes_per_step": int(n_out),
                   "output_equals_input": bool(ok),
                   "copy_only_gibs": copy_only,
                   "copy_only": "mtz_process_host in PASSTHROUGH mode on the same buffers and devices: every "
                                "byte H2D and D2H, no kernels -- what this host's PCIe / memory allows e2e",
                   "call": "mtz_process_host(pinned host stream in, pinned host stream out) on ONE handle over "
                           "%s, host wall clock around the synchronous call" % (
                               "the device group mtz_config.devices[0..%d) of a single process" % world
                               if world > 1 else "one GPU")}
            pin_out.free()
            # ---- the ring API (what js/src/binding.cc binds) on the same workload
            ring = {}
            for name, prod in (("write", "write"), ("acquire_commit", "acquire"), ("pipe", "pipe")):
                with GpuSnapshotStage("recompress", device=local, devices=devices, ring_bytes=1 << 30,
                                      out_ring_bytes=1 << 30, n_slots=4) as gr:
                    dt, ok, det = ring_run(gr, src, producer=prod, nthreads=pump_threads())
                    ok = ok and det["delivered"].get(0) == src.size and gr.end_checksum() == end_ck_of(O, end_ck, gr)
                ring[name] = {"value": round(src.size / GIB / dt, 3), "unit": "GiB/s", "ok": bool(ok),
                              "logical_gibs": round(logical / GIB / dt, 3)}
                if not ok:
                    failed.append("ring API leg %s: %s" % (name, det["errors"]))
            ring["call"] = ("write = mtz_write (one producer thread memcpy into the pinned ring); acquire_commit = "
                            "mtz_ring_acquire/commit with the slice filled by parallel memcpys (producer_alone_gibs = those "
                            "memcpys with no library behind them: the leg's ceiling on this host); pipe = read(2) "
                            "from a pipe into the slice (zfsSend.stdout shape, bound by the pipe); consumer = "
                            "mtz_out_peek/consume on the pinned output ring")
            ring["producer_alone_gibs"] = host_memcpy_ceiling(src, pump_threads())
            ring["producer_threads"] = pump_threads()
            ring["ok"] = all(v.get("ok", True) for v in ring.values() if isinstance(v, dict))
            ring["value"] = ring.get("acquire_commit", {}).get("value")
            ring["unit"] = "GiB/s"
            # ---- fan-out of the PROCESSED stream to P attached peers (configs[3]/[4])
            if world > 1:
                P = {2: 2, 4: 3, 8: 8}.get(world, min(world, 8))
                with GpuSnapshotStage("recompress", device=local, devices=devices, ring_bytes=1 << 30,
                                      out_ring_bytes=512 << 20, n_slots=4) as gf:
                    eg = [gf.fanout_attach(p) for p in range(P)]
                    dt, ok, det = ring_run(gf, src, peers=tuple(range(P)), producer="acquire",
                                           nthreads=pump_threads())
                    ok = ok and all(det["delivered"].get(p) == src.size for p in range(P))
                fan = {"peers": P, "egress_gpus": eg, "ok": bool(ok),
                       "source_once_gibs": round(total_bytes / GIB / dt, 2),
                       "delivered_gibs": round(P * total_bytes / GIB / dt, 2),
                       "delivered_logical_gibs": round(P * logical / GIB / dt, 2), "seconds": round(dt, 3),
                       "how": "one pass over the stream on %d GPUs; every batch's output crosses NVLink by one "
                              "grouped ncclBroadcast (library-owned communicator) to the egress GPUs and is "
                              "copied D2H into each peer's own pinned ring (mtz_fanout_attach / "
                              "mtz_out_peek_peer); consumers drain the rings" % world}
                if not ok:
                    failed.append("fan-out: %s" % det["errors"])
        if not args.no_cpu and world == 1:
            target = int(src.size * min(1.0, args.ref_gib * GIB / logical))
            k = int(np.searchsorted(recs_all["off"], target, side="right")) - 1
            cut = int(recs_all["off"][max(1, k)]) if k + 1 < len(recs_all) else int(src.size)
            sample = src[:cut]
            out = np.empty(sample.size + (1 << 20), dtype=np.uint8)
            n2, secs = cpu_recompress(O, sample, out, nthreads)
            n2, secs = cpu_recompress(O, sample, out, nthreads)
            O.lib().orc_mt_release()
            slog = logical * sample.size / total_bytes
            cpu = {"value": round(sample.size / GIB / secs, 3), "unit": "GiB/s", "cores": nthreads,
                   "cgroup_cpu_quota": cpu_quota(), "kind": "port",
                   "logical_gibs": round(slog / GIB / secs, 3),
                   "sample": "the first %.2f GiB of the input stream (%.2f GiB logical), second of two passes: "
                             "record-parallel oracle LZ4 decode + encode + vector Fletcher-4, sequential stamp "
                             "(oracle/mt.c)" % (sample.size / GIB, slog / GIB)}
            del out
        if world == 1 and args.verify_gib > 0:
            pin_in.free(); pin_in = None; src = None
            try:
                side = {"verify": run_verify_resident(args, O, local, min(args.steps, 20), args.warmup, peak)}
            except Exception as e:              # noqa: BLE001 -- a side workload never costs the headline line
                side = {"verify": {"error": repr(e)}}
                failed.append("side workload verify: %r" % (e,))

    if world > 1:
        dist.barrier(group=gl)
    if rank == 0:
        alg = 2.0 * total_bytes + 624.0 * len(recs_all)
        ach = alg / (k3_ms / 1e3) / 1e9 if k3_ms > 0 else None
        # which kernel the step's LZ4-encode time belongs to: the certificate (K3c) when most records
        # were proven to be the encoder's own output, the serial matcher (K3) otherwise
        certified = n_enc > 0 and n_cert >= 0.5 * n_enc
        kname = "k3c_lz4_certify" if certified else "k3_lz4_encode"
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles",
                                             "r2_k3c_traffic.json" if certified else "r2_k3_traffic.json")))
            traffic = tj.get("dram_bytes_per_algorithmic_byte") * alg / max(1.0, k3_launches)
        except Exception:
            pass
        cfg = recompress_config(total_gib)            # identical on both arms (the driver compares them)
        detail = {"records": int(len(recs_all)), "write_records": nwrites_total,
                  "stream_gib": round(total_bytes / GIB, 3), "logical_gib": round(logical / GIB, 3),
                  "ratio": round(logical / total_bytes, 3),
                  "certified_records": int(n_cert), "lz4_records_out": int(n_enc),
                  "certificate": "RECOMPRESS proves per record that the incoming LZ4 block is what the declared "
                                 "encoder emits for the decoded bytes (K3c replays the encoder's hash-table "
                                 "trajectory against the block's parse) and passes it through; records it cannot "
                                 "prove take the serial matcher; workloads.recompress_reencode_all = the same "
                                 "step with the certificate off",
                  "partition": ("record-index: %d chunks of whole records taken round-robin by %d ranks; per chunk a "
                                "40-B aggregate all-gather + the 32-B output checksum travelling the ring, "
                                "library-owned NCCL" % (4 * world, world)) if world > 1 else "single GPU",
                  "l2": "inputs_exceed_l2 (%.1f GiB per GPU >> 126 MB)" % (total_bytes / world / GIB)}
        line = {
            "metric": "snapshot_stream_gibs", "value": round(value, 3), "unit": "GiB/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u8 / u32->u64 (mod 2^64)", "data": "synthetic",
            "config": cfg, "workload_detail": detail,
            "logical_gibs": round(logical / GIB / (ms_step / 1e3), 3),
            "e2e": e2e, "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": round(ach, 1) if ach else None,
                         "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 5) if ach else None,
                         "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg / max(1.0, k3_launches),
                         "launches_per_step": int(k3_launches),
                         "k3_ms_per_step": round(k3_ms / world, 3), "codec_ms_per_step": round(codec_ms / world, 3),
                         "note": "algorithmic bytes = the fused lower bound 624 + C_in + C_out per record (SURVEY "
                                 "8d) over all records of the step / summed K3 launch time (CUDA events in the "
                                 "library, summed over ranks: K3c + K3 over the records K3c did not certify); "
                                 "both are one dependent chain of hash-table rounds per record, bound by "
                                 "instruction latency at the shared-memory occupancy limit, not by HBM"},
            "idempotent_at_full_size": same,
            "cpu_baseline": cpu, "e2e_stream_api": ring, "fanout": fan,
            "workloads": dict(side or {}, **({"recompress_reencode_all": reenc} if reenc else {})) or None,
            "clocks": clk,
            "end_checksum": ["%016x" % x for x in (end_ck or ())],
        }
        if not same:
            failed.append("RECOMPRESS output differs from the oracle-encoded input")
        if failed:
            line["failed"] = failed
        print(json.dumps(line), flush=True)
        if world > 1:
            try:
                os.unlink(shm)
            except OSError:
                pass
    if world > 1:
        dist.barrier(group=gl)
        dist.destroy_process_group()
    if pin_in is not None:
        pin_in.free()
    return 1 if failed else 0


def end_ck_of(O, resident_ck, stage):
    """END checksum the ring run must reproduce: the resident run's when it saw the END record (N=1),
    else whatever this stage reports (N>1: the resident ranks each saw a shard)."""
    return resident_ck if resident_ck is not None else stage.end_checksum()


def main():
    global RECSIZE, REC_BYTES
    args = parse_args()
    RECSIZE = args.recsize
    REC_BYTES = 312 + RECSIZE
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
