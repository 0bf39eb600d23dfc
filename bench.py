#!/usr/bin/env python
"""bench.py — audio-seconds fingerprinted per second (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this framework (CUDA, sm_100a)
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle port of the
                                                           # reference path on all host cores

A "step" = one pass of the fingerprint hot path (K1 STFT/log -> K2 peaks -> K3
hashes) over one batch of synthetic 11025 Hz mono int16 PCM.  At N=1 the batch
is BASELINE.json configs[1]: 1024 x 30 s files (density 20, fanout 3, 5
peaks/frame, 1 shift).  With N GPUs every rank fingerprints its own 1024 files
(file sharding, no data-path collective): weak scaling.

Prints ONE JSON line (rank 0).  `value` has the PCM already resident in HBM;
`e2e` goes through Analyzer.fingerprint_packed with pinned HOST buffers, the
host->device copy of the PCM and the device->host read of the hashes inside the
timed region.

--dump-outputs DIR writes what the timed steps computed in their last step as .npy
files (see dump_outputs), so that two builds can be compared output for output: the
synthetic input is a fixed function of the arguments.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SR = 11025
METRIC = "audio_seconds_fingerprinted_per_sec"
UNIT = "audio-s/s"


# ---------------------------------------------------------------- host cores
def host_cores():
    """Threads this process may really use: the scheduler affinity mask and the cgroup CPU quota
    bound it, os.cpu_count() does not (a 128-thread box with an 8-CPU quota reports 128; a pool of
    128 processes on it measured 5x below the same command on an unconstrained node, VERDICT r1)."""
    info = {"os_cpu_count": os.cpu_count() or 1}
    n = info["os_cpu_count"]
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
        n = min(n, info["affinity"])
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                quota, period = txt[0], float(txt[1])
            else:
                quota, period = txt[0], float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota not in ("max", "-1"):
                info["cgroup_cpus"] = float(quota) / period
                n = min(n, max(1, int(info["cgroup_cpus"] + 0.5)))
            break
        except (OSError, ValueError, IndexError):
            continue
    info["used"] = max(1, n)
    return info


# ---------------------------------------------------------------- synthetic input
def _gen(args):
    seed, secs = args
    from audfprint_b200.synth import synth_track
    return synth_track(seed, secs)


def make_tracks(pool, first_seed, nfiles, secs):
    return pool.map(_gen, [(first_seed + i, secs) for i in range(nfiles)], chunksize=8)


# ---------------------------------------------------------------- CPU arm (oracle)
_TRACKS = None      # set before the CPU pool is forked: workers inherit the PCM, tasks are indices


def reference_dir():
    """A checkout of the reference (dpwe/audfprint) if one is reachable: $AFP_REFERENCE or
    baseline/_ref.  It is pure Python and is NOT part of this repo; without one the CPU arm is
    the oracle port (`kind: "port"`)."""
    for d in (os.environ.get("AFP_REFERENCE"), os.path.join(ROOT, "baseline", "_ref")):
        if d and os.path.isfile(os.path.join(d, "audfprint_analyze.py")):
            return d
    return None


_REF_MOD = None


def _worker_init():
    # pay the (cold-container) import cost before anything is timed
    global _REF_MOD
    import scipy.signal  # noqa: F401
    from oracle import afp_oracle  # noqa: F401
    from audfprint_b200 import synth  # noqa: F401
    d = reference_dir()
    if d:
        sys.path.insert(0, d)
        try:
            import audfprint_analyze as ref_an       # the unmodified reference
            _REF_MOD = ref_an
        except Exception:
            _REF_MOD = None


def _cpu_fp(i):
    from audfprint_b200.synth import pcm_to_float
    d = pcm_to_float(_TRACKS[i])
    if _REF_MOD is not None:
        # Analyzer.wavfile2hashes minus the file read (audfprint_analyze.py:385-426, shifts = 1):
        # the reference's own find_peaks / peaks2landmarks / landmarks2hashes
        an = _REF_MOD.Analyzer(20.0)
        return np.asarray(_REF_MOD.landmarks2hashes(an.peaks2landmarks(an.find_peaks(d, SR))), np.int32).reshape(-1, 2)
    from oracle import afp_oracle as orc
    return orc.fingerprint(d, density=20.0, fanout=3, shifts=1)


def cpu_kind():
    return "reference" if reference_dir() else "port"


def config0_single_core(seed=0, secs=60.0, reps=5):
    """BASELINE configs[0]: one 60 s clip, single core, median of `reps` (the reference's own
    CPU path when a checkout is reachable, else the oracle port)."""
    global _TRACKS
    from audfprint_b200.synth import synth_track
    saved = _TRACKS
    _TRACKS = [synth_track(seed, secs)]
    _worker_init()
    _cpu_fp(0)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        h = _cpu_fp(0)
        ts.append(time.perf_counter() - t0)
    _TRACKS = saved
    return {"workload": "Analyzer.wavfile2hashes on one %g s 11025 Hz mono clip (BASELINE configs[0])" % secs,
            "kind": cpu_kind(), "cores": 1, "median_s": float(np.median(ts)), "runs": reps,
            "audio_s_per_s": secs / float(np.median(ts)), "hashes": int(len(h))}


def cpu_pool(tracks, nproc):
    """Fork a pool whose workers already hold `tracks` (no per-task pickling of PCM)."""
    global _TRACKS
    _TRACKS = tracks
    pool = mp.get_context("fork").Pool(nproc, initializer=_worker_init)
    pool.map(_cpu_fp, range(min(len(tracks), nproc)), chunksize=1)      # warm every worker
    return pool


def cpu_pass(pool, n):
    """Oracle port of the reference path over files 0..n-1 on the pool's processes
    (file-level parallelism, as audfprint.py:249-265 does with joblib)."""
    t0 = time.perf_counter()
    out = pool.map(_cpu_fp, range(n), chunksize=max(1, n // (8 * pool._processes)))
    return time.perf_counter() - t0, out


# ---------------------------------------------------------------- match workload (BASELINE configs[2])
_TABLE = None       # (table, counts, hashbits, depth, maxtimebits, hashesperid) for forked CPU workers
_QUERIES = None


_QTRACKS = None     # tracks the query workers cut excerpts from (set before their pool is forked)


def _gen_query(j):
    """Query j = a 10 s excerpt of track j % ntracks at a seeded offset + white noise (sigma 0.02 FS)."""
    from audfprint_b200.synth import synth_query
    trk = j % len(_QTRACKS)
    pcm, off = synth_query(_QTRACKS[trk], j, seconds=10.0, noise_sigma=0.02)
    return pcm, trk, off


def build_big_table(track_rows, track_off, nids, hashbits=20, depth=100, maxtimebits=12, seed=12345):
    """SURVEY.md §8d config 3: plant the real hashes of the queried tracks in store order,
    then fill every bucket to `depth` with uniform-random (id, time) distractors.  Returns the
    reference-format arrays; the SAME arrays feed the CPU oracle and the GPU."""
    rng = np.random.default_rng(seed)
    nb = 1 << hashbits
    ntracks = len(track_off) - 1
    ids = (np.arange(ntracks, dtype=np.int64) * (nids // ntracks))            # real tracks spread over the id space
    table = ((rng.integers(1, nids + 1, size=(nb, depth), dtype=np.int64) << maxtimebits)
             + rng.integers(0, 1292, size=(nb, depth), dtype=np.int64)).astype(np.uint32)
    h = (track_rows[:, 1].astype(np.int64)) & (nb - 1)
    t = track_rows[:, 0].astype(np.int64) & ((1 << maxtimebits) - 1)
    tid = np.repeat(ids, np.diff(track_off))
    vals = (((tid + 1) << maxtimebits) + t).astype(np.uint32)
    order = np.argsort(h, kind="stable")
    hs = h[order]
    first = np.r_[True, hs[1:] != hs[:-1]]
    start = np.maximum.accumulate(np.where(first, np.arange(len(hs)), 0))
    slot = np.arange(len(hs)) - start
    keep = slot < depth
    table[hs[keep], slot[keep]] = vals[order][keep]
    counts = np.full(nb, depth, np.int32)
    hpi = np.bincount((table >> maxtimebits).astype(np.int64).ravel() - 1, minlength=nids).astype(np.uint32)
    return table, counts, hashbits, depth, maxtimebits, hpi, ids


def _cpu_match(i):
    from oracle import afp_oracle as orc
    table, counts, hashbits, depth, mtb, hpi = _TABLE
    return orc.match_hashes(table, counts, hashbits, depth, mtb, hpi, _QUERIES[i], window=2, threshcount=5,
                            search_depth=100)


# ---------------------------------------------------------------- clocks sampler
class ClockSampler:
    """SM clock + throttle reasons polled through NVML (nvidia_ml_py) from a thread every ~2 ms
    while the timed region runs; falls back to one `nvidia-smi` query if NVML is unavailable."""

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.t = index, [], False, None
        self.max_mhz, self.h, self.nv = None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()

    def stop(self):
        if self.nv:
            self.stop_flag = True
            self.t.join(timeout=2)
            nv = self.nv
            names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown,
                     "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown,
                     "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
            reasons = sorted(n for n, bit in names.items() if any(r[1] & bit for r in self.rows))
            sm = [r[0] for r in self.rows]
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": reasons, "samples": len(sm), "source": "nvml"}
        try:
            out = subprocess.run(["nvidia-smi", "-i", str(self.index),
                                  "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.active",
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10).stdout
            f = [x.strip() for x in out.split(",")]
            return {"sm_mhz": float(f[0]), "sm_max_mhz": float(f[1]), "reasons": [f[2]], "samples": 1,
                    "source": "nvidia-smi after the timed region"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"], "samples": 0}


def warm_up(fn, min_seconds=0.7, min_calls=3):
    """Run `fn` until the GPU has been busy for min_seconds: the match legs follow CPU-only phases
    (generators, CPU baseline) during which the SM clock falls to idle (120 MHz), and a couple of
    20 ms calls are not enough to bring it back - a run of this bench measured the same kernels
    2.4x slower that way."""
    import torch
    t0 = time.perf_counter()
    n = 0
    while n < min_calls or time.perf_counter() - t0 < min_seconds:
        fn()
        n += 1
    torch.cuda.synchronize()


def bench_match(a, an, ctx, tracks, rows, roff, queries, cores, want_cpu, stream):
    """BASELINE configs[2]: 10 s noisy excerpts (4 shifts) against a 1M-id device-resident
    table (2^20 buckets x 100, every bucket full).  Reports match-only queries/s with the
    query hashes resident on the device, the same through host buffers, and audio->result."""
    global _TABLE, _QUERIES
    import torch
    from audfprint_b200 import Analyzer, HashTable, Matcher
    nq = len(queries)
    table, counts, hashbits, depth, mtb, hpi, ids = build_big_table(rows, roff, a.match_ids)
    ht = HashTable(hashbits=hashbits, depth=1, maxtime=1 << mtb)
    ht.table, ht.counts, ht.hashesperid, ht.depth = table, counts, hpi, depth
    ht.names = [None] * a.match_ids
    qan = Analyzer(device=an.device)
    qan.shifts = 4
    qpcm = [q[0] for q in queries]
    stride = (max(len(p) for p in qpcm) + 7) // 8 * 8
    hq = torch.zeros(nq * stride + 8, dtype=torch.int16).pin_memory()
    hqn = hq.numpy()
    for i, p in enumerate(qpcm):
        hqn[i * stride:i * stride + len(p)] = p
    qoffs = np.arange(nq + 1, dtype=np.int64) * stride
    qlens = np.array([len(p) for p in qpcm], np.int64)
    t0 = time.perf_counter()
    qrows, qoff = qan.fingerprint_packed(hqn, qoffs, sample_lengths=qlens)
    torch.cuda.synchronize()
    fp_s = time.perf_counter() - t0
    m = Matcher()
    m.window = 2                      # CLI default --match-win 2 (audfprint.py:363)
    res = m.match_batch(ht, (qrows, qoff))
    warm_up(lambda: m.match_batch(ht, (qrows, qoff)))
    # --- match only, host hashes in / rows out (includes H2D of the query hashes, D2H of rows)
    steps = a.steps
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = m.match_batch(ht, (qrows, qoff))
    torch.cuda.synchronize()
    host_s = (time.perf_counter() - t0) / steps
    # --- match only, query hashes resident on the device, rows left on the device
    import ctypes as C
    dq = torch.from_numpy(qrows).cuda()
    p = m._params()
    tot = C.c_int64(0)
    qoffp = np.ascontiguousarray(qoff).ctypes.data_as(C.POINTER(C.c_int64))

    def dev_step():
        ctx.check(ctx.lib.afp_match_batch(ctx.h, dq.data_ptr(), 0, nq, qoffp, C.byref(p), C.byref(tot)))
    warm_up(dev_step)
    msampler = ClockSampler(an.device if an.device is not None else 0)
    msampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        dev_step()
    e1.record(stream)
    torch.cuda.synchronize()
    mclocks = msampler.stop()
    dev_s = e0.elapsed_time(e1) * 1e-3 / steps
    st = Matcher.last_status(ht, nq)
    fast_stats = {"queries_on_fast_kernel": int(np.sum(st[:, 0] == 0)),
                  "queries_handed_to_general_kernel": int(np.sum(st[:, 0] > 0)),
                  "handover_reasons": {str(k): int(v) for k, v in zip(*np.unique(st[st[:, 0] > 0, 0], return_counts=True))},
                  "mean_multi_record_ids": float(st[:, 1].mean()), "mean_member_hits": float(st[:, 2].mean()),
                  "mean_single_record_ids_admitted": float(st[:, 3].mean()),
                  "mean_ids_above_threshcount": float(st[:, 5].mean())}
    # A/B: the general kernel alone on the same batch
    pg = m._params()
    pg.force_general = 1
    ctx.check(ctx.lib.afp_match_batch(ctx.h, dq.data_ptr(), 0, nq, qoffp, C.byref(pg), C.byref(tot)))
    torch.cuda.synchronize()
    warm_up(lambda: ctx.check(ctx.lib.afp_match_batch(ctx.h, dq.data_ptr(), 0, nq, qoffp, C.byref(pg), C.byref(tot))),
            min_seconds=0.3, min_calls=1)
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record(stream)
    for _ in range(2):
        ctx.check(ctx.lib.afp_match_batch(ctx.h, dq.data_ptr(), 0, nq, qoffp, C.byref(pg), C.byref(tot)))
    g1.record(stream)
    torch.cuda.synchronize()
    gen_s = g0.elapsed_time(g1) * 1e-3 / 2
    # --- audio -> result (fingerprint 4 shifts + match), host PCM in
    t0 = time.perf_counter()
    r2, o2 = qan.fingerprint_packed(hqn, qoffs, sample_lengths=qlens)
    res2 = m.match_batch(ht, (r2, o2))
    torch.cuda.synchronize()
    audio_s = time.perf_counter() - t0
    truth = np.array([[ids[q[1]], q[2] // 256] for q in queries])
    top = np.array([[r[0, 0], r[0, 2]] if len(r) else [-1, 0] for r in res])
    correct = int(np.sum((top[:, 0] == truth[:, 0]) & (np.abs(top[:, 1] - truth[:, 1]) <= 1)))
    nqh = int(qoff[-1])
    nprobe = 12 * nqh + 4 * nqh * depth + 28 * sum(len(r) for r in res)      # SURVEY.md §8d B_m
    out = {"metric": "match_queries_per_sec", "queries": nq, "table": "2^%d buckets x %d, %d ids, every bucket "
           "full (SURVEY.md 8d config 3)" % (hashbits, depth, a.match_ids), "query_hashes": nqh,
           "value": nq / dev_s, "unit": "queries/s", "ms_per_step": dev_s * 1e3, "clocks": mclocks,
           "e2e": {"value": nq / host_s, "unit": "queries/s", "h2d_bytes_per_step": int(qrows.nbytes + qoff.nbytes),
                   "d2h_bytes_per_step": int(sum(r.nbytes for r in res) + qoff.nbytes)},
           "audio_to_result": {"value": nq / audio_s, "unit": "queries/s",
                               "fingerprint_only_s": fp_s, "note": "10 s int16 PCM in (4 shifts) -> top rows out"},
           "roofline": {"bound": "hbm", "algorithmic_bytes_per_launch": nprobe,
                        "achieved": nprobe / dev_s / 1e9, "unit": "GB/s", "peak": measured_peaks()[0],
                        "frac": nprobe / dev_s / 1e9 / measured_peaks()[0]},
           "top1_correct": correct, "fast_kernel": fast_stats,
           "general_kernel_only": {"value": nq / gen_s, "unit": "queries/s", "ms_per_step": gen_s * 1e3},
           "cpu_baseline": None, "parity": None}
    if want_cpu:
        ns = min(a.match_cpu_sample, nq)
        _TABLE = (table, counts, hashbits, depth, mtb, hpi)
        _QUERIES = [qrows[qoff[i]:qoff[i + 1]] for i in range(ns)]
        mp_pool = mp.get_context("fork").Pool(min(cores, ns), initializer=_worker_init)
        mp_pool.map(_cpu_match, range(min(cores, ns)), chunksize=1)
        t0 = time.perf_counter()
        want = mp_pool.map(_cpu_match, range(ns), chunksize=1)
        dt = time.perf_counter() - t0
        mp_pool.close()
        bad = 0
        for i in range(ns):
            g = res[i]
            w = want[i]
            if not (g.shape == w.shape and sorted(map(tuple, g)) == sorted(map(tuple, w))):
                bad += 1
        out["cpu_baseline"] = {"value": ns / dt, "unit": "queries/s", "cores": cores, "kind": "port",
                               "sample": "%d of the %d queries, oracle port (Python loop over query hashes as "
                                         "the reference) on a %d-process pool, %.1f s wall" % (ns, nq, min(cores, ns), dt)}
        out["parity"] = {"queries_checked": ns, "queries_mismatched": bad}
    return out, res


def bench_match_sharded(a, an, rows, roff, qpool, rank, world):
    """BASELINE configs[4]: the 2^20 x 100 table sharded by track-id range over the ranks; every
    rank probes its shard for ALL queries (K4 in publish mode), packs one record per query on the
    device, ONE NCCL all-gather of the record buffers, and merges on the device
    (afp_shard_pack / afp_shard_merge).  Queries go through in batches of --match-batch."""
    import torch
    import torch.distributed as dist
    from audfprint_b200 import Analyzer, HashTable, Matcher
    from audfprint_b200 import dist as afd
    obj = [rows, roff] if rank == 0 else [None, None]
    dist.broadcast_object_list(obj, src=0)                      # table content = rank 0's hashes
    rows0, roff0 = obj
    table, counts, hashbits, depth, mtb, hpi, ids = build_big_table(rows0, roff0, a.match_ids)
    ht = HashTable(hashbits=hashbits, depth=1, maxtime=1 << mtb, device=an.device)
    ht.table, ht.counts, ht.hashesperid, ht.depth = table, counts, hpi, depth
    qan = Analyzer(device=an.device)
    qan.shifts = 4
    qh = []
    for b0 in range(0, a.match_queries, 10000):              # generate + fingerprint 10k queries at a time
        part = qpool.map(_gen_query, range(b0, min(a.match_queries, b0 + 10000)), chunksize=32)
        qh += qan.fingerprint_batch([q[0] for q in part])
        del part
    nq = len(qh)
    B = max(1, min(a.match_batch, nq))
    batches = []
    for b0 in range(0, nq, B):
        part = qh[b0:b0 + B]
        off = np.zeros(len(part) + 1, np.int64)
        off[1:] = np.cumsum([len(h) for h in part])
        batches.append((np.ascontiguousarray(np.concatenate(part)), off))
    m = Matcher()
    m.window = 2
    full = None
    if rank == 0:                                                # single-table answer for the parity check
        full = []
        for qb in batches:
            full += m.match_batch(ht, qb, sort=False)
    # ---- replicated table, queries sharded j % world (no collective): the fast layout when
    # the table fits one GPU (419 MB << 180 GB), SURVEY.md 8e
    mine = afd.shard_indices(nq, rank, world)
    my_rows = np.ascontiguousarray(np.concatenate([qh[i] for i in mine])) if len(mine) else np.zeros((0, 2), np.int32)
    my_off = np.zeros(len(mine) + 1, np.int64)
    my_off[1:] = np.cumsum([len(qh[i]) for i in mine])
    import ctypes as C
    from audfprint_b200 import _lib
    ctx = _lib.context(an.device)
    rep = m.match_batch(ht, (my_rows, my_off), sort=False)           # (uploads the table; parity below)
    dq = torch.from_numpy(my_rows).cuda()
    pp = m._params()
    tot = C.c_int64(0)
    offp = np.ascontiguousarray(my_off).ctypes.data_as(C.POINTER(C.c_int64))
    warm_up(lambda: ctx.check(ctx.lib.afp_match_batch(ctx.h, dq.data_ptr(), 0, len(mine), offp, C.byref(pp), C.byref(tot))))
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(a.steps):       # query hashes resident, rows left on the device - like the N=1 `value`
        ctx.check(ctx.lib.afp_match_batch(ctx.h, dq.data_ptr(), 0, len(mine), offp, C.byref(pp), C.byref(tot)))
    torch.cuda.synchronize()
    dtr = torch.tensor([(time.perf_counter() - t0) / a.steps], dtype=torch.float64, device="cuda")
    dist.all_reduce(dtr, op=dist.ReduceOp.MAX)
    rep_bad = 0
    if rank == 0:
        rep_bad = sum(0 if np.array_equal(rep[k], full[i]) else 1 for k, i in enumerate(mine))
    # ---- sharded table
    lo, hi = afd.id_range(a.match_ids, rank, world)
    ht.restrict_device_ids(lo, hi)
    res = None
    dbatches = [(torch.from_numpy(qb[0]).cuda(), qb[1]) for qb in batches]   # query hashes resident, like the N=1 `value`
    for k in range(24):         # collective calls: the same count on every rank; ~0.4 s of GPU work
        afd.match_sharded_batch(m, ht, dbatches[k % len(dbatches)], row_cap=16, fetch=False)
    steps = a.steps
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        for qb in dbatches:
            afd.match_sharded_batch(m, ht, qb, row_cap=16, fetch=False)      # merged rows stay on the device
    torch.cuda.synchronize()
    dt = torch.tensor([(time.perf_counter() - t0) / steps], dtype=torch.float64, device="cuda")
    dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    st = Matcher.last_status(ht, len(batches[-1][1]) - 1)
    dist.barrier()
    t0 = time.perf_counter()
    res = [afd.match_sharded_batch(m, ht, qb, row_cap=16) for qb in batches]   # host hashes in, rows out
    torch.cuda.synchronize()
    dte = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    dist.all_reduce(dte, op=dist.ReduceOp.MAX)
    out = None
    if rank == 0:
        bad, k = 0, 0
        for rws, off in res:                    # rank-order rows, ranks included: no sort on either side
            for i in range(len(off) - 1):
                bad += 0 if np.array_equal(rws[off[i]:off[i + 1]], full[k]) else 1
                k += 1
        rb = 16 + 16 * 100 + 28 * 16
        out = {"metric": "match_queries_per_sec", "queries": nq, "value": nq / float(dt[0]), "unit": "queries/s",
               "ms_per_step": float(dt[0]) * 1e3,
               "parallelism": "table sharded by track-id range x%d; every rank probes all queries; device pack, one "
                              "NCCL all-gather of %d-byte per-query records per batch of %d queries, device merge"
                              % (world, rb, B),
               "timing": "host wall clock around probe + pack + all-gather + merge, query hashes resident on the device "
                         "and merged rows left there, max over ranks (every call ends with a stream synchronise); "
                         "`e2e` = host hashes in, rows out",
               "e2e": {"value": nq / float(dte[0]), "unit": "queries/s",
                       "h2d_bytes_per_step": int(sum(b[0].nbytes + b[1].nbytes for b in batches)),
                       "d2h_bytes_per_step": int(sum(r[0].nbytes + r[1].nbytes for r in res))},
               "allgather_bytes_per_rank_per_step": int(nq * rb),
               "fast_kernel_last_batch": {"queries_on_fast_kernel": int(np.sum(st[:, 0] == 0)),
                                          "handed_to_general_kernel": int(np.sum(st[:, 0] > 0)),
                                          "mean_multi_record_ids": float(st[:, 1].mean()),
                                          "mean_single_record_ids_admitted": float(st[:, 3].mean())},
               "parity": {"queries_checked": nq, "queries_mismatched_vs_single_table": bad,
                          "compared": "rows in candidate-rank order incl. the rank column, exact"},
               "replicated_table": {"value": nq / float(dtr[0]), "unit": "queries/s", "ms_per_step": float(dtr[0]) * 1e3,
                                    "parallelism": "table replicated, queries sharded j %% %d, no collective" % world,
                                    "parity": {"queries_checked": len(mine), "queries_mismatched": rep_bad}}}
    return out


# ---------------------------------------------------------------- ingest (BASELINE configs[3])
def bench_ingest(a, rank, local_rank, world, cores, pool):
    """BASELINE configs[3]: ingest 180 s tracks, file-sharded over the ranks (track i -> rank
    i % world as audfprint.py:211-214 deals files), density 20, fanout 3, 5 peaks/frame, into a
    per-rank device-resident 2^20 x 100 table with maxtimebits 14: a step = one batch of --files
    tracks through Analyzer.fingerprint_packed + HashTable.store_batch (fingerprint AND store).
    The PCM comes from a recycled pool of --files distinct seeded tracks; every step stores them
    under new names, so the table fills (and overflows) as a real ingest does."""
    import random
    import torch
    import torch.distributed as dist
    from audfprint_b200 import Analyzer, HashTable, _lib
    nsamp = int(round(a.seconds * SR))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stride = (nsamp + 7) // 8 * 8
    # the pool of distinct tracks goes to the device chunk by chunk (4 GB of int16 PCM per rank at
    # 1024 x 180 s); only the first --e2e-files of them are also kept in pinned host memory
    dev_pcm = torch.zeros(a.files * stride + 8, dtype=torch.int16, device="cuda")
    ne2e = max(1, min(a.e2e_files, a.files))
    host_pcm = torch.zeros(ne2e * stride + 8, dtype=torch.int16).pin_memory()
    hp = host_pcm.numpy()
    for c0 in range(0, a.files, 128):
        chunk = make_tracks(pool, 10 ** 6 + rank * a.files + c0, min(128, a.files - c0), a.seconds)
        buf = np.zeros(len(chunk) * stride, np.int16)
        for i, t in enumerate(chunk):
            buf[i * stride:i * stride + nsamp] = t
            if c0 + i < ne2e:
                hp[(c0 + i) * stride:(c0 + i) * stride + nsamp] = t
        dev_pcm[c0 * stride:(c0 + len(chunk)) * stride].copy_(torch.from_numpy(buf))
    pool.close()
    offs = np.arange(a.files + 1, dtype=np.int64) * stride
    lens = np.full(a.files, nsamp, np.int64)
    offs_e, lens_e = offs[:ne2e + 1], lens[:ne2e]
    an = Analyzer(device=local_rank)
    ctx = _lib.context(local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    random.seed(1000 + rank)
    ht = HashTable(hashbits=20, depth=100, maxtime=1 << 14, device=local_rank)
    audio_s = a.files * a.seconds

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(k, pcm, o=None, ln=None):
        o, ln = (offs, lens) if o is None else (o, ln)
        an.fingerprint_packed(pcm, o, fetch=False, sample_lengths=ln)
        return ht.store_batch(["r%d/s%d/t%d" % (rank, k, i) for i in range(len(ln))])

    # parity of the first batch against the host store() (pinned to the reference), rank 0
    parity = None
    warm = max(a.warmup, 3)          # the first batches size the workspace (store scratch, overflow buffers)
    counts0 = step(-1, dev_pcm)
    if rank == 0:
        rows, roff = an.fingerprint_packed(dev_pcm, offs, sample_lengths=lens)
        random.seed(1000)
        ref = HashTable(hashbits=20, depth=100, maxtime=1 << 14, device=local_rank)
        for i in range(a.files):
            ref.store("x%d" % i, rows[roff[i]:roff[i + 1]])
        same = bool(np.array_equal(ref.counts, ht.counts) and np.array_equal(ref.table, ht.table))
        parity = {"what": "device store_batch of the first %d tracks vs the host store() of the same hashes "
                          "(bit-compatible with the reference's HashTable.store)" % a.files,
                  "tables_identical": same, "hashes": int(sum(counts0))}
    for k in range(1, warm):
        step(-1 - k, dev_pcm)
    ctx.set_profiling(True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ctx.launch_count()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fp_ms, k1_ms = 0.0, 0.0
    e0.record(stream)
    pending = None
    for k in range(a.steps):
        # as Analyzer.ingest_batch does: batch k's fingerprint kernels are launched, THEN the store of
        # batch k-1 is finished (host-side RNG replay of its overflow), THEN batch k is stored
        an.fingerprint_packed(dev_pcm, offs, fetch=False, sample_lengths=lens)
        ht.store_batch_finish(pending)
        pending = ht.store_batch_begin(["r%d/s%d/t%d" % (rank, k, i) for i in range(a.files)])
        st_ms = ctx.stage_ms()
        fp_ms += sum(st_ms[1:])
        k1_ms += st_ms[1]
    ht.store_batch_finish(pending)
    e1.record(stream)
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = ctx.launch_count() - l0
    clocks = sampler.stop()
    ctx.set_profiling(False)
    ntracks = len(ht.names)
    # end to end: pinned host PCM in every step (device calls of --e2e-files tracks)
    step(999, hp, offs_e, lens_e)
    barrier()
    t0 = time.perf_counter()
    pending = None
    for k in range(a.steps):
        an.fingerprint_packed(hp, offs_e, fetch=False, sample_lengths=lens_e)
        ht.store_batch_finish(pending)
        pending = ht.store_batch_begin(["r%d/s%d/t%d" % (rank, 1000 + k, i) for i in range(ne2e)])
    ht.store_batch_finish(pending)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([ms_total, e2e_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms = float(t[0]), float(t[1])
    nh = int(np.sum(ht.hashesperid))
    full = float(np.mean(np.minimum(ht.counts, ht.depth))) / ht.depth
    dropped = 1.0 - float(np.sum(np.minimum(ht.counts, ht.depth))) / max(1, int(np.sum(ht.counts)))
    if rank == 0:
        peak, which = measured_peaks()
        T = 1 + nsamp // 256
        k1_bytes = a.files * (2 * nsamp + 8 * 256 * T + 8 * T)
        val = audio_s * world * a.steps / (ms_total * 1e-3)
        out = {"metric": "audio_seconds_ingested_per_sec", "value": val, "unit": UNIT, "n_gpus": world,
               "steps": a.steps, "warmup": warm, "ms_per_step": ms_total / a.steps, "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
               "config": {"workload": "ingest %d x %g s synthetic tracks per GPU per step, file-sharded x%d "
                                      "(BASELINE configs[3]: 100k x 180 s over 8 GPUs = %d steps of 1024 per GPU), "
                                      "fingerprint + HashTable.store on the device, table 2^20 x 100, maxtimebits 14"
                                      % (a.files, a.seconds, world, 12),
                          "files_per_gpu_per_step": a.files, "seconds_per_file": a.seconds, "density": 20,
                          "fanout": 3, "pks_per_frame": 5, "tracks_ingested_per_gpu": ntracks,
                          "cache": "inputs larger than L2", "parallelism": "file-sharded x%d, no collective" % world},
               "clocks": clocks,
               "e2e": {"value": ne2e * a.seconds * world * a.steps / (e2e_ms * 1e-3), "unit": UNIT,
                       "files_per_device_call": ne2e,
                       "h2d_bytes_per_step": int(hp.nbytes + offs_e.nbytes + lens_e.nbytes),
                       "d2h_bytes_per_step": int(offs_e.nbytes), "ms_per_step": e2e_ms / a.steps},
               "gpu_launches": int(launches),
               "split_ms_per_step": {"fingerprint_kernels": fp_ms / a.steps, "store_and_host": ms_total / a.steps - fp_ms / a.steps},
               "roofline": {"kernel": "afp_stft_kernel<int16> (K1)", "bound": "hbm", "unit": "GB/s", "peak": peak,
                            "peak_source": which, "algorithmic_bytes_per_launch": k1_bytes, "traffic": None,
                            "launch_ms": k1_ms / a.steps, "achieved": k1_bytes / (k1_ms / a.steps * 1e-3) / 1e9,
                            "frac": k1_bytes / (k1_ms / a.steps * 1e-3) / 1e9 / peak},
               "table": {"tracks": ntracks, "hashes_stored_or_dropped": nh, "bucket_fill": full, "dropped_fraction": dropped},
               "parity": parity, "cpu_baseline": None}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    return 0


# ---------------------------------------------------------------- --dump-outputs
def fetch_last_hashes(ctx, nfiles):
    """(rows, row_offsets) of the last fingerprint batch, read back from the context's workspace
    (what Analyzer.fingerprint_packed returns with fetch=True)."""
    import ctypes as C
    roff = np.empty(nfiles + 1, np.int64)
    ctx.check(ctx.lib.afp_fetch_hashes(ctx.h, None, 1, roff.ctypes.data_as(C.POINTER(C.c_int64))))
    rows = np.empty((int(roff[-1]), 2), np.int32)
    ctx.check(ctx.lib.afp_fetch_hashes(ctx.h, rows.ctypes.data, 1, None))
    return rows, roff


def dump_outputs(d, groups, limit=64 << 20, seed=0):
    """Write ragged int results as float64 .npy files under `d` (every value is exact in float64).
    `groups` maps a name to (rows, offsets), the rows of item i (a file, a query) being
    rows[offsets[i]:offsets[i + 1]].  A group gives d/<name>.npy (the rows of the items written,
    one item after the other), d/<name>_offsets.npy and d/<name>_items.npy (the item indices).
    All items are written when the files fit in `limit` bytes; otherwise every group is cut to
    a seeded random sample of whole items, the same for the same arguments, that fits."""
    os.makedirs(d, exist_ok=True)
    rng = np.random.default_rng(seed)
    sizes = {name: 8 * (rows.size + 2 * len(off)) for name, (rows, off) in groups.items()}
    total = sum(sizes.values())
    for name, (rows, off) in groups.items():
        off = np.asarray(off, np.int64)
        lens = np.diff(off)
        items = np.arange(len(lens))
        if total > limit:
            order = rng.permutation(len(lens))
            cost = np.cumsum(8 * (lens[order] * rows.shape[1] + 2))
            budget = (limit - 3 * 128 * len(groups)) * sizes[name] // total - 8     # 128-byte .npy headers
            items = np.sort(order[cost <= budget])
        n = lens[items]
        start = np.cumsum(n) - n
        idx = np.repeat(off[items], n) + np.arange(int(n.sum())) - np.repeat(start, n)
        np.save(os.path.join(d, name + ".npy"), rows[idx].astype(np.float64))
        np.save(os.path.join(d, name + "_offsets.npy"), np.concatenate([[0], np.cumsum(n)]).astype(np.float64))
        np.save(os.path.join(d, name + "_items.npy"), items.astype(np.float64))


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 10; 12 with --config 3)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--files", type=int, default=1024, help="files per GPU per step")
    ap.add_argument("--seconds", type=float, default=None, help="seconds per file (default 30; 180 with --config 3)")
    ap.add_argument("--cpu-sample", type=int, default=512, help="files in the CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true",
                    help="profiling aid: run only the device-resident timed region (e2e = null)")
    ap.add_argument("--match-queries", type=int, default=None,
                    help="queries of the match workload (0 = skip; default 10000 = BASELINE configs[2]; "
                         "100000 with --config 4)")
    ap.add_argument("--match-ids", type=int, default=1000000)
    ap.add_argument("--e2e-files", type=int, default=256, help="--config 3: tracks per device call of the host-PCM leg")
    ap.add_argument("--match-batch", type=int, default=10000, help="queries per device call of the sharded match")
    ap.add_argument("--config", type=int, default=1, choices=[1, 2, 3, 4],
                    help="BASELINE.json configs[]: 1 batch fingerprint (default; the driver's line), 2 match 10k "
                         "queries on 1 GPU, 3 ingest 180 s tracks incl. store, 4 sharded-table match of 100k queries")
    ap.add_argument("--match-cpu-sample", type=int, default=1024,
                    help="queries in the CPU baseline / parity sample of the match leg (~3 s on 16 cores)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the hashes (and match rows) of the last timed step as .npy files under DIR")
    a = ap.parse_args()
    if a.match_queries is None:
        a.match_queries = 100000 if a.config == 4 else 10000
    if a.steps is None:
        a.steps = 12 if a.config == 3 else 10
    if a.seconds is None:
        a.seconds = 180.0 if a.config == 3 else 30.0
    if a.dump_outputs and (a.impl == "reference" or a.config in (3, 4)):
        ap.error("--dump-outputs writes the outputs of --config 1 and 2 of this implementation")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores_info = host_cores()
    cores = cores_info["used"]
    if a.impl != "reference":
        cores = max(2, cores // max(1, world))      # every rank forks its own generator pool
    nsamp = int(round(a.seconds * SR))
    config = {"workload": "batch fingerprint %d x %g s synthetic 11025 Hz mono int16 files per GPU "
                          "(BASELINE configs[1])" % (a.files, a.seconds),
              "files_per_gpu": a.files, "seconds_per_file": a.seconds, "sr": SR, "density": 20, "fanout": 3,
              "pks_per_frame": 5, "shifts": 1,
              "cache": "inputs larger than L2 (%.0f MB int16 PCM + %.1f GB FP64 log-spectrogram per step)"
                       % (a.files * nsamp * 2 / 1e6, a.files * (1 + nsamp // 256) * 2048 / 1e9),
              "parallelism": "file-sharded x%d, no collective" % world}

    # worker pools are forked BEFORE torch/CUDA is touched
    pool = mp.get_context("fork").Pool(cores, initializer=_worker_init)

    # ------------------------------------------------------------ reference arm
    if a.impl == "reference":
        if rank != 0:
            return 0
        # 16 files per worker per step: enough tasks that the pool's tail imbalance stays small
        per_step = min(max(cores * 16, 128), a.files)
        tracks = make_tracks(pool, 0, per_step, a.seconds)
        pool.close()
        cpool = cpu_pool(tracks, cores)
        for _ in range(min(a.warmup, 1)):
            cpu_pass(cpool, per_step)
        times = []
        for _ in range(a.steps):
            dt, _ = cpu_pass(cpool, per_step)
            times.append(dt)
        tot = sum(times)
        val = per_step * a.seconds * a.steps / tot
        kind = cpu_kind()
        sample = "%d of the %d files per step, %s over a %d-process pool (affinity/cgroup-limited: %s)" % (
            per_step, a.files, "the unmodified reference (find_peaks/peaks2landmarks/landmarks2hashes)"
            if kind == "reference" else "oracle port (NumPy/SciPy, same call structure as the reference)",
            cores, cores_info)
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus,
                          "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * tot / a.steps,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                          "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind,
                                           "sample": sample, "host_cores": cores_info},
                          "config0": config0_single_core(),
                          "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    # ------------------------------------------------------------ our arm
    if a.config == 3:
        return bench_ingest(a, rank, local_rank, world, cores, pool)
    tracks = make_tracks(pool, rank * a.files, a.files, a.seconds)
    do_match = a.match_queries > 0
    queries, qpool = None, None
    if do_match:
        # queries are excerpts of RANK 0's tracks (a sharded table is the same table on every rank);
        # their pool is forked now (before CUDA is touched) with those tracks in memory, and asked for
        # the queries batch by batch: 100k x 10 s of PCM never exist at once
        global _QTRACKS
        _QTRACKS = tracks if rank == 0 else make_tracks(pool, 0, a.files, a.seconds)
        qpool = mp.get_context("fork").Pool(cores)
        if world == 1:
            queries = qpool.map(_gen_query, range(a.match_queries), chunksize=32)
    pool.close()
    want_cpu = rank == 0 and world == 1 and not a.no_cpu_baseline
    cpool = cpu_pool(tracks[:min(a.cpu_sample, a.files)], cores) if want_cpu else None

    import torch
    import torch.distributed as dist
    from audfprint_b200 import Analyzer, _lib
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    # pack: every file starts on a 16-byte boundary (TMA staging of interior tiles)
    stride = (nsamp + 7) // 8 * 8
    host_pcm = torch.zeros(a.files * stride + 8, dtype=torch.int16).pin_memory()
    hp = host_pcm.numpy()
    for i, t in enumerate(tracks):
        hp[i * stride:i * stride + nsamp] = t
    offs = np.arange(a.files + 1, dtype=np.int64) * stride
    lens = np.full(a.files, nsamp, np.int64)
    dev_pcm = host_pcm.cuda(non_blocking=False)
    audio_s = a.files * a.seconds

    an = Analyzer(device=local_rank)
    ctx = _lib.context(local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)        # kernels + our timing events on the same stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        an.fingerprint_packed(dev_pcm, offs, fetch=False, sample_lengths=lens)

    for _ in range(max(a.warmup, 3)):
        step_resident()
    torch.cuda.synchronize()

    # ---- device-resident timing (value) + live per-stage timing (roofline) ----------------
    ctx.set_profiling(True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = ctx.launch_count()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stages = np.zeros(5)
    e0.record(stream)
    for _ in range(a.steps):
        step_resident()
        stages += np.array(ctx.stage_ms())
    e1.record(stream)
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = ctx.launch_count() - l0
    clocks = sampler.stop()
    ctx.set_profiling(False)
    stages /= a.steps
    last_step = fetch_last_hashes(ctx, a.files) if a.dump_outputs and rank == 0 else None

    # ---- end to end: pinned host PCM in, hashes + offsets out, every step --------------------
    rows, roff = an.fingerprint_packed(dev_pcm, offs, sample_lengths=lens)
    nhash = int(roff[-1])
    e2e_s = float("nan")
    if not a.no_e2e:
        host_rows = torch.empty((nhash + 1024, 2), dtype=torch.int32).pin_memory()
        hr = host_rows.numpy()
        for _ in range(2):
            an.fingerprint_packed(hp, offs, sample_lengths=lens, host_rows=hr)
        barrier()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            r2, o2 = an.fingerprint_packed(hp, offs, sample_lengths=lens, host_rows=hr)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        assert int(o2[-1]) == nhash and np.array_equal(r2, rows)

    # ---- opt-in FP32 spectrogram mode (secondary; the headline stays FP64 / bit-identical) ----
    fp32 = None
    if rank == 0:
        an32 = Analyzer(device=local_rank)
        an32.precision = "fp32"
        r32, o32 = an32.fingerprint_packed(dev_pcm, offs, sample_lengths=lens)
        for _ in range(3):
            an32.fingerprint_packed(dev_pcm, offs, fetch=False, sample_lengths=lens)
        torch.cuda.synchronize()
        ctx.set_profiling(True)
        st32 = np.zeros(5)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        for _ in range(a.steps):
            an32.fingerprint_packed(dev_pcm, offs, fetch=False, sample_lengths=lens)
            st32 += np.array(ctx.stage_ms())
        f1.record(stream)
        torch.cuda.synchronize()
        ctx.set_profiling(False)
        st32 /= a.steps
        ms32 = f0.elapsed_time(f1) / a.steps
        differ = sum(0 if np.array_equal(rows[roff[i]:roff[i + 1]], r32[o32[i]:o32[i + 1]]) else 1
                     for i in range(a.files))
        k64 = set(map(tuple, np.column_stack([np.repeat(np.arange(a.files), np.diff(roff)), rows]).tolist()))
        k32 = set(map(tuple, np.column_stack([np.repeat(np.arange(a.files), np.diff(o32)), r32]).tolist()))
        T_ = 1 + nsamp // 256
        b32 = a.files * (2 * nsamp + 4 * 256 * T_ + 8 * T_)
        pk, which_ = measured_peaks()
        fp32 = {"note": "Analyzer.precision='fp32': FP32 STFT+log, float spectrogram; NOT the headline "
                        "(hashes are not guaranteed bit-identical)",
                "value": audio_s / (ms32 * 1e-3), "unit": UNIT, "ms_per_step": ms32,
                "stages_ms": {"k1_stft_log": float(st32[1]), "stats": float(st32[2]), "k2_peaks": float(st32[3]),
                              "k3_hashes": float(st32[4])},
                "roofline": {"kernel": "afp_stft_f32_kernel<int16>", "bound": "hbm",
                             "algorithmic_bytes_per_launch": b32, "achieved": b32 / (st32[1] * 1e-3) / 1e9,
                             "unit": "GB/s", "peak": pk, "peak_source": which_,
                             "frac": b32 / (st32[1] * 1e-3) / 1e9 / pk},
                "vs_fp64": {"files": a.files, "files_with_any_difference": differ,
                            "hashes_fp64": len(k64), "hashes_fp32": len(k32),
                            "jaccard": len(k64 & k32) / max(1, len(k64 | k32))}}
        an._configure(1)        # back to the FP64 tables for whatever follows

    t = torch.tensor([ms_total, e2e_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms = float(t[0]), float(t[1])

    # ---- CPU baseline on a bounded sample + parity spot check (rank 0, N=1 only) -------------
    cpu = None
    parity = None
    if want_cpu:
        ns = min(a.cpu_sample, a.files)
        dt, want = cpu_pass(cpool, ns)
        bad = sum(0 if np.array_equal(rows[roff[i]:roff[i + 1]], want[i]) else 1 for i in range(ns))
        parity = {"files_checked": ns, "files_mismatched": bad,
                  "hashes_checked": int(sum(len(w) for w in want))}
        cpu = {"value": ns * a.seconds / dt, "unit": UNIT, "cores": cores, "kind": cpu_kind(),
               "host_cores": cores_info,
               "sample": "%d of the %d files (%.0f audio-s), %s on a %d-process pool, %.1f s wall"
                         % (ns, a.files, ns * a.seconds, "reference" if cpu_kind() == "reference" else "oracle port",
                            cores, dt)}

    # ---- BASELINE configs[0] through the drop-in call: Analyzer.wavfile2hashes on ONE 60 s WAV file
    # (one file per device call - the reference's own usage pattern), median of 7
    config0 = None
    if rank == 0:
        import tempfile
        import wave
        from audfprint_b200.synth import synth_track
        clip = synth_track(0, 60.0)
        with tempfile.TemporaryDirectory() as td:
            fn = os.path.join(td, "clip60.wav")
            with wave.open(fn, "wb") as w:
                w.setnchannels(1); w.setsampwidth(2); w.setframerate(SR)
                w.writeframes(clip.tobytes())
            an0 = Analyzer(device=local_rank)
            h0 = an0.wavfile2hashes(fn)
            ts = []
            for _ in range(7):
                t0 = time.perf_counter()
                h0 = an0.wavfile2hashes(fn)
                ts.append(time.perf_counter() - t0)
        config0 = {"workload": "Analyzer.wavfile2hashes on one 60 s 11025 Hz mono WAV (BASELINE configs[0]), file read "
                               "+ host->device + K1..K3 + hashes back, one file per device call",
                   "median_s": float(np.median(ts)), "runs": 7, "audio_s_per_s": 60.0 / float(np.median(ts)),
                   "hashes": int(len(h0))}
        if want_cpu:
            from oracle import afp_oracle as orc
            from audfprint_b200.synth import pcm_to_float
            config0["identical_to_cpu_path"] = bool(np.array_equal(h0, orc.fingerprint(pcm_to_float(clip))))
            config0["cpu_single_core"] = config0_single_core()

    match, match_rows = None, None
    if do_match and world == 1:
        match, match_rows = bench_match(a, an, ctx, tracks, rows, roff, queries, cores, want_cpu, stream)
    elif do_match:
        match = bench_match_sharded(a, an, rows, roff, qpool, rank, world)

    if rank == 0:
        peak, which = measured_peaks()
        T = 1 + nsamp // 256
        k1_bytes = a.files * (2 * nsamp + 8 * 256 * T + 8 * T)      # int16 PCM in, FP64 logs + nyq out
        k1_ms = float(stages[1])
        achieved = k1_bytes / (k1_ms * 1e-3) / 1e9
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "k1_traffic.json")) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
        except Exception:
            pass
        out = {"metric": METRIC, "value": audio_s * world * a.steps / (ms_total * 1e-3), "unit": UNIT,
               "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_total / a.steps,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
               "data": "synthetic", "config": config, "clocks": clocks,
               "e2e": None if a.no_e2e else
               {"value": audio_s * world * a.steps / (e2e_ms * 1e-3), "unit": UNIT,
                "h2d_bytes_per_step": int(hp.nbytes + offs.nbytes + lens.nbytes),
                "d2h_bytes_per_step": int(nhash * 8 + roff.nbytes + 8),
                "ms_per_step": e2e_ms / a.steps},
               "gpu_launches": int(launches),
               "roofline": {"kernel": "afp_stft_kernel<int16> (K1: frame+window+512-pt real FFT+log|.|, FP64)",
                            "bound": "hbm", "achieved": achieved, "peak": peak, "peak_source": which,
                            "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                            "traffic_source": "dram__bytes_read+write of one launch, ncu --set full capture "
                                              "profiles/r01_v5_k1_stft.txt (K1 is unchanged since)",
                            "algorithmic_bytes_per_launch": k1_bytes, "launch_ms": k1_ms},
               "stages_ms": {"h2d": float(stages[0]), "k1_stft_log": float(stages[1]),
                             "stats": float(stages[2]), "k2_peaks": float(stages[3]),
                             "k3_hashes": float(stages[4])},
               "hashes_per_step": nhash, "cpu_baseline": cpu, "parity": parity, "config0": config0,
               "match": match, "fp32_mode": fp32}
        if a.config in (2, 4) and match is not None:
            # BASELINE configs[2] / configs[4]: the match leg is the headline line, the fingerprint
            # numbers of the same run ride along
            line = dict(match)
            line.update({"n_gpus": world, "steps": a.steps, "warmup": 2, "higher_is_better": True,
                         "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "u32",
                         "data": "synthetic", "clocks": clocks, "gpu_launches": 2,
                         "config": {"workload": ("match %d x 10 s noisy synthetic queries (4 shifts) against a "
                                                 "%d-track device-resident HashTable 2^20 x 100 (BASELINE configs[%d])"
                                                 % (a.match_queries, a.match_ids, a.config)) +
                                    (", table sharded by id range x%d, one NCCL all-gather per batch" % world
                                     if world > 1 else ""),
                                    "cache": "419 MB table + per-query scratch larger than L2 in aggregate"},
                         "fingerprint_leg": {k: out[k] for k in ("value", "unit", "ms_per_step", "stages_ms")}})
            print(json.dumps(line))
        else:
            print(json.dumps(out))
    if last_step is not None:
        groups = {"hashes": last_step}                  # (time, hash) rows of every file
        if match_rows is not None:                      # (id, count, offset, ...) rows of every query
            groups["match_rows"] = (np.concatenate(match_rows).reshape(-1, 7),
                                    np.concatenate([[0], np.cumsum([len(r) for r in match_rows])]))
        dump_outputs(a.dump_outputs, groups)
    if world > 1:
        dist.destroy_process_group()
    if cpool:
        cpool.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
