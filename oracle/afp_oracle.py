"""CPU oracle for the landmark-fingerprint hot path.  TEST INFRASTRUCTURE ONLY.

This module is a NumPy restatement of the reference algorithm (dpwe/audfprint
@ cb03ba99) for the one path SURVEY.md §8 scopes: STFT -> log-magnitude ->
onset high-pass -> decaying-threshold peak picking (forward + backward) ->
landmark pairing -> 20-bit hash packing -> bucketed hash probe -> per-track
time-offset histogram matching.

Rules of use (see the task's parity section):
  * only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s CPU-baseline /
    `--impl reference` legs may import it, and only as the checker / baseline;
  * the product (`audfprint_b200/`) never imports it and has no CPU fallback.

Pinning: the reference ships no numeric known-answer tests for this path
(SURVEY.md §4, §8c).  The oracle is therefore pinned against OUTPUTS OF THE LIVE
REFERENCE, imported from /root/reference in the build container by
`oracle/make_golden.py`, committed as `tests/golden/*.npz`;
`tests/test_oracle_golden.py` checks this module against them bit-for-bit.

Third-party arithmetic the reference leans on (not under /root/reference,
un-pinned in requirements.txt:1-2): numpy (pocketfft `rfft`, `log`, `exp`,
`mean`) and `scipy.signal.lfilter`.  The oracle calls the same numpy routines
and restates lfilter's direct-form-II-transposed recurrence explicitly.

Every function cites the reference file:line it follows.
"""
from __future__ import annotations

import numpy as np

# ---- constants (audfprint_analyze.py:55-78, 125-151) -----------------------
N_FFT = 512
N_HOP = 256
HPF_POLE = 0.98
F1_BITS, DF_BITS, DT_BITS = 8, 6, 6


def decay_constant(density: float, n_hop: int = N_HOP) -> float:
    """Masking-envelope decay per frame.  audfprint_analyze.py:277 (OVERSAMP=1)."""
    return float((1 - 0.01 * (density * np.sqrt(n_hop / 352.8) / 35)) ** (1 / 1))


def analysis_window(n_fft: int = N_FFT) -> np.ndarray:
    """Symmetric Hann of n_fft+2 points with the zero end points dropped.
    audfprint_analyze.py:279."""
    return np.hanning(n_fft + 2)[1:-1]


def gaussian_table(npoints: int, width: float) -> np.ndarray:
    """E[j] = exp(-0.5*((j - npoints)/width)^2), j = 0..2*npoints.
    audfprint_analyze.py:187-192."""
    return np.exp(-0.5 * ((np.arange(-npoints, npoints + 1) / width) ** 2))


# ---- K1: STFT + conditioning -------------------------------------------------
def stft_complex(d: np.ndarray, n_fft: int = N_FFT, n_hop: int = N_HOP) -> np.ndarray:
    """Reflect-pad n_fft/2, frame with hop n_hop, window, real FFT; returns the
    complex (n_fft/2+1, T) array.  stft.py:62-94 as called from
    audfprint_analyze.py:279-282."""
    win = analysis_window(n_fft)
    padded = np.pad(d, n_fft // 2, mode="reflect")                 # stft.py:88
    nfr = 1 + (len(padded) - n_fft) // n_hop                       # stft.py:33
    gather = (np.arange(nfr) * n_hop)[:, None] + np.arange(n_fft)[None, :]
    frames = padded[gather] * win                                  # stft.py:93 (f32*f64 -> f64)
    return np.fft.rfft(frames, n_fft).transpose()                  # stft.py:94


def hpf_rows(x: np.ndarray, pole: float = HPF_POLE, explicit: bool = False) -> np.ndarray:
    """Per-row lfilter([1,-1],[1,-pole]) with zero initial state, in
    scipy's direct-form-II-transposed order: y = z + x ; z = -x + pole*y.
    audfprint_analyze.py:293-295.  When scipy is importable the same C routine
    the reference calls is used (one call over all rows); the explicit
    recurrence below is bit-identical to it (tests/test_oracle_golden.py)."""
    if not explicit:
        try:
            import scipy.signal
            return scipy.signal.lfilter([1, -1], [1, -pole], x, axis=1)
        except ImportError:
            pass
    rows, cols = x.shape
    y = np.empty_like(x)
    z = np.zeros(rows, dtype=x.dtype)
    for t in range(cols):
        xt = x[:, t]
        yt = z + xt
        z = -xt + pole * yt
        y[:, t] = yt
    return y


def conditioned_sgram(d: np.ndarray):
    """|STFT| -> log with floor max/1e6 -> minus global mean -> HPF -> drop the
    Nyquist row.  Returns (sgram (256,T) float64, mag (257,T) float64).
    audfprint_analyze.py:280-295."""
    mag = np.abs(stft_complex(d))
    smax = np.max(mag)
    if smax > 0.0:
        s = np.log(np.maximum(mag, smax / 1e6))
        s = s - np.mean(s)
    else:
        s = mag                                                    # all-zero input: :287-290
    return hpf_rows(s)[:-1, :], mag


# ---- K2: peak picking --------------------------------------------------------
def local_max_mask(v: np.ndarray) -> np.ndarray:
    """v[i] is a local max iff v[i] >= v[i-1] (or i == 0) and v[i+1] < v[i]
    (or i == n-1).  audfprint_analyze.py:36-52."""
    n = len(v)
    ge_left = np.ones(n + 1, dtype=bool)
    ge_left[1:n] = v[1:] >= v[:-1]
    ge_left[n] = False
    return ge_left[:n] & ~ge_left[1:]


def spread_local_maxes(v: np.ndarray, etab: np.ndarray) -> np.ndarray:
    """max over local maxima k of v[k]*E(i - k), starting from zeros.
    audfprint_analyze.py:153-197."""
    n = len(v)
    out = np.zeros(n)
    for k in np.nonzero(local_max_mask(v))[0]:
        out = np.maximum(out, v[k] * etab[n - k: 2 * n - k])
    return out


def forward_prune(sgram: np.ndarray, a_dec: float, etab: np.ndarray, maxpks: int):
    """Forward decaying-threshold pass.  Returns per-column lists of
    (value, bin) in the order they were accepted (value desc, bin desc on
    ties).  audfprint_analyze.py:199-231."""
    nb, T = sgram.shape
    thr = spread_local_maxes(np.max(sgram[:, :min(10, T)], axis=1), etab)
    accepted = []
    for t in range(T):
        col = sgram[:, t]
        cand = np.nonzero(local_max_mask(col) & (col > thr))[0]
        ranked = sorted(((col[b], int(b)) for b in cand), reverse=True)[:maxpks]
        for val, b in ranked:
            thr = np.maximum(thr, val * etab[nb - b: 2 * nb - b])
        accepted.append(ranked)
        thr = thr * a_dec
    return accepted


def backward_prune(sgram: np.ndarray, accepted, a_dec: float, etab: np.ndarray):
    """Backward pass over the forward peaks.  Returns a bool mask (256,T).
    audfprint_analyze.py:233-253."""
    nb, T = sgram.shape
    keep = np.zeros((nb, T), dtype=bool)
    for t, lst in enumerate(accepted):
        for _, b in lst:
            keep[b, t] = True
    thr = spread_local_maxes(sgram[:, -1], etab)
    for t in range(T - 1, -1, -1):
        for val, b in accepted[t]:                # already (value, bin) descending
            if val >= thr[b]:
                thr = np.maximum(thr, val * etab[nb - b: 2 * nb - b])
                if t + 1 < T:
                    keep[b, t + 1] = False        # same bin, following column
            else:
                keep[b, t] = False
        thr = a_dec * thr
    return keep


def find_peaks(d: np.ndarray, density: float = 20.0, f_sd: float = 30.0, maxpks: int = 5):
    """PCM (float) -> list of (col, bin), column-major, bins ascending.
    audfprint_analyze.py:255-308."""
    if len(d) == 0:
        return []
    sgram, _ = conditioned_sgram(d)
    etab = gaussian_table(sgram.shape[0], f_sd)
    a_dec = decay_constant(density)
    acc = forward_prune(sgram, a_dec, etab, maxpks)
    keep = backward_prune(sgram, acc, a_dec, etab)
    cols, bins = np.nonzero(keep.T)
    return list(zip(cols.tolist(), bins.tolist()))


# ---- K3: pairing + hashing ---------------------------------------------------
def peaks_to_landmarks(pklist, fanout: int = 3, mindt: int = 2, targetdt: int = 63, targetdf: int = 31):
    """Each peak pairs with the first `fanout` later peaks having
    col2 in [col+mindt, min(scols, col+targetdt)) and |bin2-bin| < targetdf,
    visited column-ascending then bin-ascending.  audfprint_analyze.py:310-343."""
    out = []
    if not len(pklist):
        return out
    scols = pklist[-1][0] + 1
    by_col = [[] for _ in range(scols)]
    for c, b in pklist:
        by_col[c].append(b)
    for c in range(scols):
        for b in by_col[c]:
            got = 0
            for c2 in range(c + mindt, min(scols, c + targetdt)):
                if got >= fanout:
                    break
                for b2 in by_col[c2]:
                    if abs(b2 - b) < targetdf and got < fanout:
                        out.append((c, b, b2, c2 - c))
                        got += 1
    return out


def landmarks_to_hashes(lms) -> np.ndarray:
    """(col, bin1, bin2, dt) -> int32 rows [col, bin1:8 | df:6 | dt:6].
    audfprint_analyze.py:81-96."""
    a = np.array(lms, dtype=np.int64).reshape(-1, 4)
    out = np.zeros((a.shape[0], 2), dtype=np.int32)
    if a.shape[0]:
        out[:, 0] = a[:, 0]
        out[:, 1] = (((a[:, 1] & 0xFF) << (DF_BITS + DT_BITS))
                     | (((a[:, 2] - a[:, 1]) & 0x3F) << DT_BITS)
                     | (a[:, 3] & 0x3F))
    return out


def hashes_to_landmarks(hashes):
    """Inverse of landmarks_to_hashes with sign-extended df.
    audfprint_analyze.py:99-112."""
    res = []
    for t, h in hashes:
        dt = h & 0x3F
        b1 = (h >> 12) & 0xFF
        df = (h >> 6) & 0x3F
        if df >= 32:
            df -= 64
        res.append((int(t), int(b1), int(b1 + df), int(dt)))
    return res


def shift_offsets(shifts: int, n_hop: int = N_HOP):
    """Sample offsets of the sub-frame shifts.  audfprint_analyze.py:374-376."""
    return [int(s / shifts * n_hop) for s in range(shifts)]


def fingerprint(d: np.ndarray, density: float = 20.0, fanout: int = 3, shifts: int = 1,
                f_sd: float = 30.0, maxpks: int = 5, mindt: int = 2, targetdt: int = 63,
                targetdf: int = 31) -> np.ndarray:
    """PCM (float) -> int32 (U,2) rows [time, hash], sorted by (time, hash),
    duplicates across shifts removed.  audfprint_analyze.py:369-377, 401-422.
    mindt / targetdt / targetdf are the Analyzer attributes of the pairing window (:139-143).
    Returns an empty (0,2) array where the reference returns [] (:401-402)."""
    lists = []
    if shifts < 2:
        lists.append(find_peaks(d, density, f_sd, maxpks))
    else:
        for off in shift_offsets(shifts):
            lists.append(find_peaks(d[off:], density, f_sd, maxpks))
    if shifts < 2 and len(lists[0]) == 0:
        return np.zeros((0, 2), np.int32)
    rows = np.concatenate([landmarks_to_hashes(peaks_to_landmarks(pl, fanout, mindt, targetdt, targetdf))
                           for pl in lists])
    key = (rows[:, 0].astype(np.uint64) << np.uint64(32)) + rows[:, 1].astype(np.uint64)
    key = np.unique(key)
    return np.stack([key >> np.uint64(32), key & np.uint64(0xFFFFFFFF)], axis=1).astype(np.int32)


# ---- hash table --------------------------------------------------------------
class Table:
    """Fixed-size bucketed table: `table` uint32 (2^hashbits, depth), `counts`
    int32 (2^hashbits).  Entry = ((id+1) << maxtimebits) + (time & mask).
    hash_table.py:59-81, 91-138."""

    def __init__(self, hashbits=20, depth=100, maxtimebits=14):
        self.hashbits, self.depth, self.maxtimebits = hashbits, depth, maxtimebits
        self.table = np.zeros((1 << hashbits, depth), np.uint32)
        self.counts = np.zeros(1 << hashbits, np.int32)
        self.hashesperid = np.zeros(0, np.uint32)
        self.names = []

    def store(self, name, rows, rng=None):
        """Insert rows [time, hash] for a new/known name.  On bucket overflow
        the reference draws `random.randint(0, count)` (hash_table.py:127-131);
        pass `rng` (an object with .randint(a, b) inclusive) to reproduce it."""
        if name not in self.names:
            self.names.append(name)
            self.hashesperid = np.append(self.hashesperid, np.uint32(0))
        id_ = self.names.index(name)
        hmask = (1 << self.hashbits) - 1
        tmask = (1 << self.maxtimebits) - 1
        idval = (id_ + 1) << self.maxtimebits
        for t, h in rows:
            h = int(h) & hmask
            cnt = int(self.counts[h])
            val = idval + (int(t) & tmask)
            if cnt < self.depth:
                self.table[h, cnt] = val
            else:
                slot = rng.randint(0, cnt)
                if slot < self.depth:
                    self.table[h, slot] = val
            self.counts[h] = cnt + 1
        self.hashesperid[id_] += len(rows)


def get_hits(table: np.ndarray, counts: np.ndarray, hashbits: int, depth: int, maxtimebits: int,
             q: np.ndarray) -> np.ndarray:
    """Query rows [time, hash] -> int32 (nhits,4) rows [id, dtime, hash, qtime]
    in (query row, slot) order.  hash_table.py:150-176."""
    q = np.asarray(q).reshape(-1, 2)
    hmask = (1 << hashbits) - 1
    tmask = (1 << maxtimebits) - 1
    chunks = []
    for t, h in q:
        b = int(h) & hmask
        n = min(depth, int(counts[b]))
        v = table[b, :n].astype(np.int64)
        blk = np.empty((n, 4), np.int32)
        blk[:, 0] = (v >> maxtimebits) - 1
        blk[:, 1] = (v & tmask) - int(t)
        blk[:, 2] = b
        blk[:, 3] = int(t)
        chunks.append(blk)
    if not chunks:
        return np.zeros((0, 4), np.int32)
    return np.concatenate(chunks, axis=0)


# ---- K4: matching ------------------------------------------------------------
def rank_candidates(hits: np.ndarray, hashesperid: np.ndarray, threshcount: int, search_depth: int):
    """Distinct ids ordered by raw/hashesperid descending, truncated to
    min(#ids with raw > threshcount, search_depth).  audfprint_match.py:124-147.

    Tie rule: the reference reverses an UNSTABLE argsort (:139), so the order
    of equal weighted counts is implementation-defined there.  The oracle (and
    the CUDA path) define it: equal weights -> larger id first, which is what
    reversing a stable ascending argsort gives."""
    ids, raw = np.unique(hits[:, 0], return_counts=True)
    wtd = raw / hashesperid[ids].astype(float)
    order = np.argsort(wtd, kind="stable")[::-1]
    depth = min(int(np.count_nonzero(raw > threshcount)), search_depth)
    order = order[:depth]
    return ids[order], raw[order]


def offset_histogram_rows(hits: np.ndarray, ids, raws, window: int, threshcount: int,
                          max_alignments_per_id: int = 100) -> np.ndarray:
    """Per candidate id: histogram of dtime, keep local maxima, repeatedly take
    the first arg-max while it is > threshcount, report the +-window sum.
    Rows [id, count, dtime, raw, rank, 0, 0].  audfprint_match.py:241-312
    (find_time_range off)."""
    rows = []
    if hits.shape[0] == 0:
        return np.zeros((0, 7), np.int32)
    tmin = int(np.min(hits[:, 1]))
    for rank, (id_, raw) in enumerate(zip(ids, raws)):
        dts = hits[hits[:, 0] == id_, 1].astype(np.int64) - tmin
        bc = np.bincount(dts)
        lm = np.where(local_max_mask(bc), bc, 0).astype(np.float64)
        found = 0
        while True:
            mode = int(np.argmax(lm))
            if lm[mode] <= threshcount:
                break
            lo, hi = max(0, mode - window), mode + window + 1
            rows.append([int(id_), int(np.sum(bc[lo:hi])), mode + tmin, int(raw), rank, 0, 0])
            lm[lo:hi] = 0
            found += 1
            if found > max_alignments_per_id:
                break
    return np.array(rows, dtype=np.int32).reshape(-1, 7)


def support_rows(hits: np.ndarray, id_: int, mode: int, window: int) -> np.ndarray:
    """Hits of one id within +-window of an offset, in query-time order
    (the selection of audfprint_match.py:163-165 and :184-188)."""
    h = hits[np.argsort(hits[:, 3], kind="stable")]
    return h[(h[:, 0] == id_) & (np.abs(h[:, 1].astype(np.int64) - mode) <= window)]


def time_range(hits: np.ndarray, id_: int, mode: int, window: int, quantile: float = 0.02):
    """Quantile-trimmed first / last query time supporting an alignment
    (audfprint_match.py:173-195)."""
    t = support_rows(hits, id_, mode, window)[:, 3]
    n = len(t)
    return int(t[int(n * quantile)]), int(t[int(n * (1.0 - quantile)) - 1])


def pair_bits(hits: np.ndarray) -> int:
    """Bits the reference reserves for the query time when packing (time, hash)
    pairs - encpowerof2(max time), at least 1 (audfprint_match.py:46-48,157)."""
    return max(1, int(np.ceil(np.log(max(1, int(np.max(hits[:, 3])))) / np.log(2))))


def matching_pairs(hits: np.ndarray, id_: int, mode: int, window: int) -> np.ndarray:
    """Distinct (query time, hash) pairs behind one alignment, as the reference packs
    and unpacks them (audfprint_match.py:149-171) - int64 (n,2)."""
    bits = pair_bits(hits)
    sup = support_rows(hits, id_, mode, window)
    packed = sorted(set(int(t) + (int(h) << bits) for t, h in zip(sup[:, 3], sup[:, 2])))
    return np.array([[v & ((1 << bits) - 1), v >> bits] for v in packed], np.int64).reshape(-1, 2)


def exact_rows(hits: np.ndarray, ids, raws, window: int, threshcount: int,
               find_time_range: bool = False, quantile: float = 0.02) -> np.ndarray:
    """exact_count branch (audfprint_match.py:197-239): every local maximum >= threshcount of a
    candidate's offset histogram is an alignment; its count is the number of distinct
    (query time, hash) pairs within +-window."""
    rows = []
    for rank, (id_, raw) in enumerate(zip(ids, raws)):
        dts = hits[hits[:, 0] == id_, 1].astype(np.int64)
        base = int(dts.min())
        hist = np.bincount(dts - base)
        for k in np.nonzero(local_max_mask(hist) & (hist >= threshcount))[0]:
            mode = int(k) + base
            n = len(matching_pairs(hits, id_, mode, window))
            if n >= threshcount:
                lo, hi = time_range(hits, id_, mode, window, quantile) if find_time_range else (0, 0)
                rows.append([int(id_), n, mode, int(raw), rank, lo, hi])
    return np.array(rows, dtype=np.int32).reshape(-1, 7)


def match_hashes(table, counts, hashbits, depth, maxtimebits, hashesperid, q,
                 window=1, threshcount=5, search_depth=100, max_alignments_per_id=100,
                 exact_count=False, find_time_range=False, quantile=0.02, hashesfor=None):
    """get_hits -> rank_candidates -> offset_histogram_rows (or exact_rows) -> sort by count
    descending (stable; the reference's final argsort, audfprint_match.py:335,
    is unstable so equal counts are implementation-defined there).
    With hashesfor=k also returns the matching pairs of sorted row k (:347-352)."""
    hits = get_hits(table, counts, hashbits, depth, maxtimebits, q)
    if hits.shape[0] == 0:
        return np.zeros((0, 7), np.int32)
    ids, raws = rank_candidates(hits, hashesperid, threshcount, search_depth)
    if exact_count:
        rows = exact_rows(hits, ids, raws, window, threshcount, find_time_range, quantile)
    else:
        rows = offset_histogram_rows(hits, ids, raws, window, threshcount, max_alignments_per_id)
        if find_time_range:
            for r in rows:
                r[5], r[6] = time_range(hits, int(r[0]), int(r[2]), window, quantile)
    rows = rows[np.argsort(-rows[:, 1], kind="stable")]
    if hashesfor is None:
        return rows
    return rows, matching_pairs(hits, int(rows[hashesfor, 0]), int(rows[hashesfor, 2]), window)
