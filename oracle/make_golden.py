"""Generate tests/golden/*.npz by running the LIVE reference (read-only at
/root/reference) on the deterministic cases of tests/cases.py.

Run in the build container only (the GPU box has no /root/reference):
    python oracle/make_golden.py

Only OUTPUT ARRAYS of the reference are stored; no reference source is copied.
The reference's file reader is replaced by an in-memory PCM provider because
the image has neither ffmpeg nor a working WAV fallback (SURVEY.md §8c).
"""
from __future__ import annotations

import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = os.environ.get("AFP_REFERENCE", "/root/reference")
sys.path.insert(0, REF)

import audfprint_analyze as ref_an      # noqa: E402  (the reference)
import audfprint_match as ref_ma        # noqa: E402
import audio_read as ref_ar             # noqa: E402
import hash_table as ref_ht             # noqa: E402

from audfprint_b200.synth import synth_track, pcm_to_float     # noqa: E402
from tests import cases                                        # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
_PCM = {}


def _fake_reader(filename, sr=None, channels=None):
    return pcm_to_float(_PCM[filename]), 11025


ref_ar.audio_read = _fake_reader
SG_STRIDE = 97


def run_analyzer(pcm, density=20.0, fanout=3, capture=False):
    """Reference find_peaks / peaks2landmarks / landmarks2hashes on one PCM."""
    an = ref_an.Analyzer(density)
    an.maxpairsperpeak = fanout
    grabbed = {}
    if capture:
        orig = an._decaying_threshold_fwd_prune

        def spy(sgram, a_dec):
            grabbed["sgram"] = np.array(sgram)
            return orig(sgram, a_dec)
        an._decaying_threshold_fwd_prune = spy
    d = pcm_to_float(pcm)
    pk = an.find_peaks(d, 11025)
    lm = an.peaks2landmarks(pk)
    hs = ref_an.landmarks2hashes(lm)
    return an, pk, lm, hs, grabbed.get("sgram")


def file_hashes(pcm, shifts, density=20.0, fanout=3):
    an = ref_an.Analyzer(density)
    an.maxpairsperpeak = fanout
    an.shifts = shifts
    _PCM["x"] = pcm
    h = an.wavfile2hashes("x")
    return np.asarray(h, dtype=np.int32).reshape(-1, 2)


def main():
    os.makedirs(OUT, exist_ok=True)
    g = {}
    import stft as ref_stft
    for name, seed, secs in cases.NOISE_CASES:
        pcm = synth_track(seed, secs)
        an, pk, lm, hs, sg = run_analyzer(pcm, capture=True)
        g[name + "/peaks"] = np.array(pk, np.int32).reshape(-1, 2)
        g[name + "/landmarks"] = np.array(lm, np.int32).reshape(-1, 4)
        g[name + "/hashes"] = hs
        g[name + "/sgram_cols"] = sg[:, ::SG_STRIDE].copy()
        mag = np.abs(ref_stft.stft(pcm_to_float(pcm), n_fft=512, hop_length=256,
                                   window=np.hanning(514)[1:-1]))
        g[name + "/mag_cols"] = mag[:, ::SG_STRIDE].copy()
        g[name + "/wf2h_s1"] = file_hashes(pcm, 1)
        g[name + "/wf2h_s4"] = file_hashes(pcm, 4)
        print(name, "peaks", len(pk), "hashes", len(hs), "s4", len(g[name + "/wf2h_s4"]))
    for name in cases.ADVERSARIAL:
        pcm = cases.adversarial_pcm(name)
        _, pk, _, _, _ = run_analyzer(pcm)
        g[name + "/peaks"] = np.array(pk, np.int32).reshape(-1, 2)
        g[name + "/wf2h_s1"] = file_hashes(pcm, 1)
        g[name + "/wf2h_s4"] = file_hashes(pcm, 4)
        print(name, "N", len(pcm), "peaks", len(pk), "s1", len(g[name + "/wf2h_s1"]),
              "s4", len(g[name + "/wf2h_s4"]))
    for name, seed, secs, dens, fan in cases.DENSITY_CASES:
        pcm = synth_track(seed, secs)
        _, pk, _, _, _ = run_analyzer(pcm, dens, fan)
        g[name + "/peaks"] = np.array(pk, np.int32).reshape(-1, 2)
        g[name + "/wf2h_s1"] = file_hashes(pcm, 1, dens, fan)
        print(name, "peaks", len(pk), "s1", len(g[name + "/wf2h_s1"]))
    np.savez_compressed(os.path.join(OUT, "fingerprint.npz"), **g)

    # ---- small databases: store / get_hits / match_hashes ---------------------
    m = {}
    track_hashes = [file_hashes(cases.db_track(i), 1) for i in range(cases.DB_NTRACKS)]
    for i, h in enumerate(track_hashes):
        m["track%d/hashes" % i] = h
    queries = {}
    for j in range(cases.DB_QUERIES):
        for tag, sigma in (("clean", 0.0), ("noisy", 0.02)):
            pcm, trk, off = cases.db_query(j, sigma)
            key = "q%d_%s" % (j, tag)
            queries[key] = file_hashes(pcm, 4)
            m[key + "/q"] = queries[key]
            m[key + "/truth"] = np.array([trk, off], np.int32)
    # db: roomy 2^20 table;  db2: 2^12 buckets x 8 so that hashes alias and
    # buckets overflow (reservoir replacement, counts > depth)
    for db, (hashbits, depth) in {"db": (cases.DB_HASHBITS, cases.DB_DEPTH),
                                  "db2": (cases.DB2_HASHBITS, cases.DB2_DEPTH)}.items():
        random.seed(1234)                  # reference store() draws from the global RNG
        ht = ref_ht.HashTable(hashbits=hashbits, depth=depth, maxtime=1 << cases.DB_MAXTIMEBITS)
        for i, h in enumerate(track_hashes):
            ht.store("track%d" % i, h)
        nz = np.nonzero(ht.counts)[0]
        m[db + "/params"] = np.array([hashbits, depth, cases.DB_MAXTIMEBITS], np.int32)
        m[db + "/buckets"] = nz.astype(np.int32)
        m[db + "/counts"] = ht.counts[nz]
        m[db + "/rows"] = ht.table[nz]
        m[db + "/hashesperid"] = np.asarray(ht.hashesperid)
        print(db, ": buckets", len(nz), "overfull", int(np.sum(ht.counts > ht.depth)))
        for cfg, (window, thresh, sdepth) in {"a": (2, 5, 100), "b": (1, 2, 3)}.items():
            mt = ref_ma.Matcher()
            mt.window, mt.threshcount, mt.search_depth = window, thresh, sdepth
            m["cfg_%s" % cfg] = np.array([window, thresh, sdepth], np.int32)
            for key, q in queries.items():
                hits = ht.get_hits(q)
                rows = mt.match_hashes(ht, q)
                if cfg == "a":
                    m["%s/%s/hits" % (db, key)] = hits
                m["%s/%s/rows_%s" % (db, key, cfg)] = rows
                # tie diagnostics: is the order of candidates / rows well defined?
                ids, raw = np.unique(hits[:, 0], return_counts=True)
                wtd = raw / ht.hashesperid[ids].astype(float)
                dep = min(int(np.count_nonzero(raw > thresh)), sdepth)
                srt = np.sort(wtd)[::-1][:dep + 1]
                tie_w = bool(dep and np.any(srt[:-1] == srt[1:]))
                tie_c = bool(len(np.unique(rows[:, 1])) != len(rows))
                m["%s/%s/ties_%s" % (db, key, cfg)] = np.array([tie_w, tie_c])
                print(db, cfg, key, "nq", len(q), "hits", len(hits), "nrows", len(rows),
                      "top", rows[:1].tolist(), "truth", m[key + "/truth"][0],
                      m[key + "/truth"][1] // 256, "ties", tie_w, tie_c)
    # the hits go to a file of their own, column-major (it compresses better), so that each
    # file stays under 1 MB; tests.conftest.load_golden joins the two
    np.savez_compressed(os.path.join(OUT, "match_hits.npz"),
                        **{k: np.asfortranarray(v) for k, v in m.items() if k.endswith("/hits")})
    np.savez_compressed(os.path.join(OUT, "match.npz"), **{k: v for k, v in m.items() if not k.endswith("/hits")})

    # a small database saved by the reference's own HashTable.save (gzip pickle of the object,
    # hash_table.py:178-197): the mirror class must load it (tests/test_abi_cpu.py)
    random.seed(99)
    small = ref_ht.HashTable(hashbits=10, depth=4, maxtime=1 << 10)
    for i in range(6):
        small.store("ref_track%d" % i, track_hashes[i][:120])
    small.params["samplerate"] = 11025
    small.save(os.path.join(OUT, "ref_db.pklz"))
    np.savez_compressed(os.path.join(OUT, "ref_db_arrays.npz"), table=small.table, counts=small.counts,
                        hashesperid=np.asarray(small.hashesperid))


if __name__ == "__main__":
    main()
