"""GPU: K3 (afp_landmark_kernel, afp_merge_kernel, afp_landmarks_from_peaks) at the limits of the
parameters it accepts and past 2^20 columns, against the oracle.  tests/test_oracle_pairing.py pins the
oracle to the reference on the same inputs."""
import ctypes as C
import os

import numpy as np
import pytest

from audfprint_b200 import Analyzer
from audfprint_b200.synth import synth_track, pcm_to_float
from oracle import afp_oracle as orc
from tests import cases
from tests.conftest import GOLDEN

pytestmark = pytest.mark.gpu

MERGE_SLOTS = 256   # AFP_MAX_MERGE: hash slots of one (file, column) over all shifts


@pytest.fixture(scope="module")
def golden_pairing():
    return np.load(os.path.join(GOLDEN, "pairing.npz"))


def analyzer(mindt, targetdt, targetdf, fanout, maxpks, shifts=1, density=20.0, f_sd=30.0):
    an = Analyzer(density=density)
    an.mindt, an.targetdt, an.targetdf, an.maxpairsperpeak = mindt, targetdt, targetdf, fanout
    an.maxpksperframe, an.shifts, an.f_sd = maxpks, shifts, f_sd
    return an


def device_peaks(an, shift, nfiles):
    """Peaks of one shift of every file of the last batch, as int32 (n, 2) arrays."""
    ctx = an._configure(an.shifts)
    poff = np.empty(nfiles + 1, np.int64)
    ctx.check(ctx.lib.afp_fetch_peaks(ctx.h, shift, None, 1, poff.ctypes.data_as(C.POINTER(C.c_int64))))
    rows = np.empty((int(poff[-1]), 2), np.int32)
    ctx.check(ctx.lib.afp_fetch_peaks(ctx.h, shift, rows.ctypes.data, 1, None))
    return [rows[poff[i]:poff[i + 1]] for i in range(nfiles)]


def hashes_of_peaks(peak_lists, a, b, fanout, mindt=2, targetdt=63, targetdf=31):
    """The oracle's rows with time in [a, b) for one file, from its peak list of every shift.  They depend
    only on the peaks in columns [a, b + targetdt), so only those are paired."""
    rows = []
    for pk in peak_lists:
        sub = pk[(pk[:, 0] >= a) & (pk[:, 0] < b + targetdt)]
        lms = orc.peaks_to_landmarks([(int(c) - a, int(v)) for c, v in sub], fanout, mindt, targetdt, targetdf)
        h = orc.landmarks_to_hashes(lms)
        h[:, 0] += a
        rows.append(h[h[:, 0] < b])
    rows = np.concatenate(rows)
    key = np.unique((rows[:, 0].astype(np.uint64) << np.uint64(32)) + rows[:, 1].astype(np.uint64))
    return np.stack([key >> np.uint64(32), key & np.uint64(0xFFFFFFFF)], axis=1).astype(np.int32).reshape(-1, 2)


def edges(rows):
    """(dt, df) of every hash row."""
    h = rows[:, 1].astype(np.int64)
    df = (h >> 6) & 0x3F
    return h & 0x3F, np.where(df >= 32, df - 64, df)


@pytest.mark.parametrize("k", range(len(cases.PAIRING_SETTINGS)))
def test_pairing_settings_vs_oracle(golden_pairing, k):
    """fingerprint_batch with mindt / targetdt / targetdf / fanout / maxpks / shifts at the limits the
    analyzer accepts, bit for bit against the oracle; each setting reaches the edges it is there for."""
    mindt, targetdt, targetdf, fanout, maxpks, shifts, density, f_sd = cases.PAIRING_SETTINGS[k]
    tracks = cases.pairing_tracks()
    an = analyzer(mindt, targetdt, targetdf, fanout, maxpks, shifts, density, f_sd)
    got = an.fingerprint_batch(tracks)
    pks = [device_peaks(an, s, len(tracks)) for s in range(shifts)]
    full, merged, dts, dfs, selfpair, samecol = False, 0, set(), set(), False, False
    for i, (t, g) in enumerate(zip(tracks, got)):
        d = pcm_to_float(t)
        want = orc.fingerprint(d, density=density, fanout=fanout, shifts=shifts, f_sd=f_sd, maxpks=maxpks,
                               mindt=mindt, targetdt=targetdt, targetdf=targetdf)
        assert np.array_equal(g, want), i
        assert np.array_equal(g, golden_pairing["h/%d/%d" % (k, i)]), i
        assert np.array_equal(pks[0][i], golden_pairing["p/%d/%d" % (k, i)]), i
        per_col = np.zeros(len(t) // 256 + 1, np.int64)     # hash slots filled per column, all shifts
        for s in range(shifts):
            pk = pks[s][i]
            full |= bool(len(pk)) and np.bincount(pk[:, 0]).max() == maxpks
            lms = np.array(orc.peaks_to_landmarks([tuple(r) for r in pk.tolist()], fanout, mindt, targetdt,
                                                  targetdf), np.int64).reshape(-1, 4)
            np.add.at(per_col, lms[:, 0], 1)
        merged = max(merged, int(per_col.max()))
        dt, df = edges(g)
        dts |= set(dt.tolist())
        dfs |= set(np.abs(df).tolist())
        selfpair |= bool(np.any((dt == 0) & (df == 0)))
        samecol |= bool(np.any((dt == 0) & (df != 0)))
    assert full, "no column holds maxpks peaks"
    assert {mindt, targetdt - 1} <= dts and max(dts) == targetdt - 1 and min(dts) == mindt
    assert targetdf - 1 in dfs and max(dfs) == targetdf - 1
    if mindt == 0:
        assert selfpair and samecol
    if shifts * maxpks * fanout == MERGE_SLOTS:
        assert merged == MERGE_SLOTS, merged          # the merge buffer filled up


@pytest.mark.parametrize("m", range(len(cases.PEAK_LIST_SETTINGS)))
def test_peaks2landmarks_past_2_20_columns(golden_pairing, m):
    """Explicit peak lists starting at columns 0, 2^20 - 300, 2^20 + 1000, 2^21 + 5 and 2^22 - 100: the
    same landmarks in the same order as the oracle and the reference."""
    mindt, targetdt, targetdf, fanout, maxpks = cases.PEAK_LIST_SETTINGS[m]
    an = analyzer(mindt, targetdt, targetdf, fanout, maxpks)
    for j, start in enumerate(cases.PEAK_LIST_STARTS):
        pk = golden_pairing["lists/%d/%d/peaks" % (m, j)]
        got = an.peaks2landmarks([tuple(r) for r in pk.tolist()])
        # the oracle's pairing only depends on column differences: run it from column 0
        want = [(c + start, b1, b2, dt) for c, b1, b2, dt in
                orc.peaks_to_landmarks([(c - start, b) for c, b in pk.tolist()], fanout, mindt, targetdt, targetdf)]
        assert got == want, (m, start)
        assert np.array_equal(np.array(got, np.int32).reshape(-1, 4),
                              golden_pairing["lists/%d/%d/landmarks" % (m, j)]), (m, start)


@pytest.mark.parametrize("shifts", [1, 4])
def test_file_longer_than_2_20_frames(shifts):
    """(2^20 + 3000) frames of int16 next to a short file (>= 64 MB of host PCM: the chunked copy path).
    The hashes with times in [0, 2000), [2^20 - 5000, 2^20 + 5000) and the last 300 columns are the
    oracle's pairing, hashing and de-duplication of the device's own peaks of every shift."""
    n = ((1 << 20) + 3000) * 256
    long_pcm = np.resize(synth_track(7300, 60.0), n)
    short = synth_track(7301, 7.0)
    an = Analyzer()
    an.shifts = shifts
    got = an.fingerprint_batch([long_pcm, short])
    assert np.array_equal(got[1], orc.fingerprint(pcm_to_float(short), shifts=shifts))
    pks = [device_peaks(an, s, 2)[0] for s in range(shifts)]
    T = 1 + n // 256
    t = got[0][:, 0]
    assert t.max() >= T - 64 and np.all(np.diff(t) >= 0)
    for a, b in ((0, 2000), ((1 << 20) - 5000, (1 << 20) + 5000), (T - 300, T)):
        want = hashes_of_peaks(pks, a, b, an.maxpairsperpeak)
        assert len(want) > 0
        assert np.array_equal(got[0][(t >= a) & (t < b)], want), (a, b)


def test_bad_pairing_parameters_are_rejected():
    """Out-of-range pairing windows and more than 256 merge slots raise; the context stays usable."""
    sig = synth_track(7400, 5.0)
    want = orc.fingerprint(pcm_to_float(sig))
    an = Analyzer()
    assert np.array_equal(an.fingerprint_batch([sig])[0], want)
    pk = [(0, 10), (3, 20), (5, 12)]
    for bad in (dict(targetdt=65), dict(targetdf=0), dict(targetdf=33), dict(mindt=-1), dict(mindt=63),
                dict(maxpksperframe=1, maxpairsperpeak=257), dict(maxpksperframe=1, maxpairsperpeak=1, shifts=257)):
        b = Analyzer()
        for attr, v in bad.items():
            setattr(b, attr, v)
        with pytest.raises(Exception):
            b.fingerprint_batch([sig])
        if "shifts" not in bad:      # peaks2landmarks pairs one list: it runs at one shift
            with pytest.raises(Exception):
                b.peaks2landmarks(pk)
        # the configuration in place before the failed call, then a different valid one
        assert np.array_equal(an.fingerprint_batch([sig])[0], want), bad
    c = analyzer(0, 64, 32, 4, 5)
    assert c.peaks2landmarks(pk) == orc.peaks_to_landmarks(pk, 4, 0, 64, 32)
    assert np.array_equal(c.fingerprint_batch([sig])[0],
                          orc.fingerprint(pcm_to_float(sig), fanout=4, mindt=0, targetdt=64, targetdf=32))


def test_unpadded_packing_vs_oracle():
    """fingerprint_packed with offsets = cumsum(lengths): files start anywhere, so K1 stages them through
    its scalar path.  int16 and float32, host and device-resident PCM, 1 and 4 shifts."""
    import torch
    sigs = [synth_track(7500 + i, 2.0 + 0.61 * i)[: 20001 + 4099 * i] for i in range(5)]
    lens = np.array([len(s) for s in sigs], np.int64)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    assert np.any(off[1:-1] % 8 != 0) and np.any(off[1:-1] % 4 != 0)
    an = Analyzer()
    for shifts in (1, 4):
        want = [orc.fingerprint(pcm_to_float(s), shifts=shifts) for s in sigs]
        for pcm in (np.concatenate(sigs), pcm_to_float(np.concatenate(sigs))):
            for where in ("host", "device"):
                buf = pcm if where == "host" else torch.from_numpy(pcm).cuda()
                rows, roff = an.fingerprint_packed(buf, off, shifts)
                for i, w in enumerate(want):
                    assert np.array_equal(rows[roff[i]:roff[i + 1]], w), (shifts, pcm.dtype, where, i)
