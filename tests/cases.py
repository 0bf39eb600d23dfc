"""Deterministic input cases shared by oracle/make_golden.py and the tests.

Every case is reproducible from its name alone, so the golden fixtures only
need to store the reference's OUTPUTS.
"""
from __future__ import annotations

import numpy as np

from audfprint_b200.synth import synth_track, synth_query, SR

# (name, seed, seconds)
NOISE_CASES = [("s%d_%ds" % (seed, secs), seed, secs)
               for seed in (0, 1, 2) for secs in (10, 30, 60)]


def adversarial_pcm(name: str) -> np.ndarray:
    """int16 PCM for the edge cases SURVEY.md §8c lists."""
    if name == "zeros":                      # identically zero signal
        return np.zeros(3 * SR, np.int16)
    if name == "silence_gap":                # 3 s of exact digital silence inside a track
        x = synth_track(7, 12.0).copy()
        x[4 * SR:7 * SR] = 0
        return x
    if name.startswith("short"):             # N <= n_fft: multi-bounce reflection
        n = int(name[5:])
        return synth_track(11, 1.0)[:n].copy()
    if name == "ragged":                     # N not a multiple of the hop
        return synth_track(5, 10.0)[:100003].copy()
    if name == "sine":                       # constant-amplitude sine (plateaus / exact ties)
        t = np.arange(8 * SR)
        return np.round(8000 * np.sin(2 * np.pi * 1000.0 * t / SR)).astype(np.int16)
    if name == "square":                     # clipped periodic signal
        t = np.arange(6 * SR)
        return (12000 * np.sign(np.sin(2 * np.pi * 441.0 * t / SR))).astype(np.int16)
    if name == "impulses":                   # sparse clicks over digital silence
        x = np.zeros(6 * SR, np.int16)
        x[::3001] = 20000
        return x
    raise KeyError(name)


ADVERSARIAL = ["zeros", "silence_gap", "short1", "short2", "short100", "short256", "short257",
               "short300", "short511", "short512", "short513", "ragged", "sine", "square",
               "impulses"]

DENSITY_CASES = [("s3_20s_d70", 3, 20, 70.0, 8), ("s3_20s_d100", 3, 20, 100.0, 10),
                 ("s4_20s_d7", 4, 20, 7.0, 3)]   # (name, seed, secs, density, fanout)

# small database used for the probe / match goldens
DB_NTRACKS = 40
DB_TRACK_SECONDS = 20.0
DB_QUERIES = 12          # query j is cut from track (j * 3) % DB_NTRACKS
DB_DEPTH = 20            # small depth so that some buckets overflow
DB_HASHBITS = 20
DB_MAXTIMEBITS = 14
DB2_HASHBITS = 12         # aliasing + overflowing buckets (cf. Makefile:83-85 hashbits=16)
DB2_DEPTH = 8


def db_track(i: int) -> np.ndarray:
    return synth_track(100 + i, DB_TRACK_SECONDS)


def db_query(j: int, noise_sigma: float = 0.01):
    trk = (j * 3) % DB_NTRACKS
    pcm, off = synth_query(db_track(trk), j, seconds=10.0, noise_sigma=noise_sigma)
    return pcm, trk, off

# host-side table bookkeeping sequence (oracle/make_golden_table_ops.py)
TABLE_OPS_SEED = 2718
TABLE_OPS_HASHBITS = 10
TABLE_OPS_DEPTH = 6
TABLE_OPS_ROWS = 600

# configs[3] / configs[2] geometry (oracle/make_golden_long.py): 180 s tracks, a table whose
# 12 time bits alias for them (95 s), 10 s and 200 s queries (the latter > 21k hashes at 4 shifts)
LONG_SECONDS = 180.0
LONG_SEEDS = [300, 301, 302]
LONG_HASHBITS = 16
LONG_DEPTH = 20
LONG_MAXTIMEBITS = 12
LONG_QUERIES = [(0, 10.0), (1, 10.0), (2, 10.0), (1, 170.0)]      # (track index, seconds)

# K3 pairing window at its limits (oracle/make_golden_pairing.py, tests/test_gpu_landmarks.py).
# (mindt, targetdt, targetdf, fanout, maxpks, shifts, density, f_sd); densities are high enough that
# columns fill up to maxpks peaks
PAIRING_SETTINGS = [
    (0, 63, 31, 3, 5, 1, 20.0, 30.0),       # same-column pairs and self-pairs
    (0, 64, 32, 16, 16, 1, 1000.0, 3.0),    # both 6-bit fields at their limit; merge buffer full
    (0, 64, 32, 4, 16, 4, 2000.0, 2.0),     # merge buffer full across shifts
    (2, 63, 31, 1, 16, 16, 1000.0, 3.0),    # 16 shifts
    (63, 64, 32, 2, 8, 2, 60.0, 30.0),      # only dt = 63
    (1, 3, 4, 2, 5, 4, 40.0, 30.0),         # narrowest useful window
    (5, 20, 10, 4, 8, 3, 40.0, 30.0),       # 3 shifts: int16 shift items start off 16-byte boundaries
]
PAIRING_SEED = 7113
PAIRING_SECONDS = 8.0


def gapped_track(seed: int, seconds: float) -> np.ndarray:
    """synth_track with digital silence of 40..63 frames between bursts of 4..29 frames: isolated
    peak clusters whose pairs span the whole pairing window."""
    x = synth_track(seed, seconds).copy()
    rng = np.random.default_rng(seed + 1)
    c = int(rng.integers(20, 40))
    while c * 256 < len(x):
        g = int(rng.integers(40, 64))
        x[c * 256:(c + g) * 256] = 0
        c += g + int(rng.integers(4, 30))
    return x


def pairing_tracks():
    """The two int16 tracks every pairing setting is run on."""
    return [synth_track(PAIRING_SEED, PAIRING_SECONDS), gapped_track(PAIRING_SEED, PAIRING_SECONDS)]


# explicit peak lists for peaks2landmarks: (mindt, targetdt, targetdf, fanout, maxpks), and first columns
# on both sides of 2^20, 2^21 and 2^22
PEAK_LIST_SETTINGS = [(2, 63, 31, 3, 5), (0, 64, 32, 8, 16)]
PEAK_LIST_STARTS = [0, (1 << 20) - 300, (1 << 20) + 1000, (1 << 21) + 5, (1 << 22) - 100]
PEAK_LIST_COLUMNS = 400


def peak_list(seed: int, start: int, maxpks: int, ncols: int = PEAK_LIST_COLUMNS) -> np.ndarray:
    """int32 (n, 2) rows (col, bin), column-major, bins ascending, in columns [start, start + ncols):
    full columns of maxpks peaks, empty stretches longer than any pairing window, and a lone final
    peak after a gap."""
    rng = np.random.default_rng(seed)
    counts = rng.integers(0, maxpks + 1, ncols)
    counts[rng.random(ncols) < 0.15] = maxpks
    for g0 in (ncols // 4, ncols // 2 + 13):
        counts[g0:g0 + 70 + int(rng.integers(0, 10))] = 0
    counts[ncols - 40:] = 0
    counts[0] = maxpks
    counts[-1] = 1
    rows = [(start + c, int(b)) for c in range(ncols)
            for b in np.sort(rng.choice(256, int(counts[c]), replace=False))]
    return np.array(rows, np.int32).reshape(-1, 2)
