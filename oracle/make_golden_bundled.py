"""Golden vectors from the reference's OWN bundled test material
(/root/reference/tests/data: Nine_Lives/*.mp3 + query.mp3), i.e. what the
reference's Makefile exercises (`make test_onecore`: new / add / match at
--density 100, Makefile:12-29), produced by the LIVE reference.

BASELINE.json's north_star asks for "match results bit-identical to the
reference on the bundled tests/data queries"; round 1 recorded that as blocked
(no MP3 decoder in the image).  oracle/ffdecode.py decodes the files through
the FFmpeg libraries vendored with OpenCV, with the parameters of the
reference's `ffmpeg -f s16le -ac 1 -ar 11025` pipe (audio_read.py:196-203), and
the live reference runs on that PCM with its reader replaced by the decoder.

Run in the build container only (the GPU box has no /root/reference):
    python oracle/make_golden_bundled.py
Stored in tests/golden/bundled.npz: reference OUTPUTS (hashes, table rows,
match rows, report lines); in tests/golden/bundled_pcm.npz: the decoded int16
PCM of the query and of PCM_TRACKS (the input the GPU parity tests need, where
neither the MP3s nor the reference are at hand).  No reference source is copied.
"""
from __future__ import annotations

import glob
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

from oracle import ffdecode             # noqa: E402
from tests.conftest import option_ties  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "bundled.npz")
DATA = os.path.join(REF, "tests", "data")
DENSITIES = (100.0, 20.0)               # the Makefile's setting, the CLI default
PCM_TRACKS = (0, 4, 8, 12)              # tracks whose PCM is committed (0-based)
# name -> Matcher settings on top of the CLI defaults (audfprint.py:303-317)
MATCH_CONFIGS = {
    "default": {},
    "top5": {"max_returns": 5},
    "exact": {"max_returns": 5, "exact_count": True},
    "range": {"max_returns": 5, "find_time_range": True},
    "exact_range_time": {"max_returns": 5, "exact_count": True, "find_time_range": True, "sort_by_time": True},
    "tight": {"max_returns": 3, "window": 1, "threshcount": 2, "search_depth": 4},
}

_PCM = {}


def _reader(filename, sr=None, channels=None):
    """Stands where the reference's ffmpeg pipe stands (audio_read.py:56-99)."""
    return _PCM[filename].astype(np.float32) / 32768.0, 11025


ref_ar.audio_read = _reader


def track_files():
    return sorted(glob.glob(os.path.join(DATA, "Nine_Lives", "*.mp3")))


def short(path):
    return os.path.relpath(path, DATA)


def excerpt(pcm):
    """The 5 s of a track that start 3 s in (also used by the tests)."""
    return pcm[3 * 11025:8 * 11025].copy()


def make_analyzer(density, shifts):
    """audfprint.py:280-299 with the command line's defaults."""
    an = ref_an.Analyzer()
    an.density = density
    an.maxpksperframe = 5
    an.maxpairsperpeak = 3
    an.f_sd = 30.0
    an.shifts = shifts
    an.target_sr = 11025
    an.n_fft = 512
    an.n_hop = 256
    return an


def make_matcher(**kw):
    """audfprint.py:303-317 with the command line's defaults, then the overrides."""
    mt = ref_ma.Matcher()
    mt.window, mt.threshcount, mt.max_returns, mt.search_depth = 2, 5, 1, 100
    mt.sort_by_time = mt.exact_count = mt.find_time_range = False
    mt.verbose = True
    mt.time_quantile = 0.05
    for k, v in kw.items():
        setattr(mt, k, v)
    return mt


def main():
    files = track_files()
    query = os.path.join(DATA, "query.mp3")
    assert len(files) == 13 and os.path.isfile(query)
    for f in files + [query]:
        _PCM[short(f)] = ffdecode.decode(f)
    g = {"names": np.array([short(f) for f in files]), "query_name": np.array(short(query)),
         "query/pcm": _PCM[short(query)]}
    for k in PCM_TRACKS:
        g["track%d/pcm" % k] = _PCM[short(files[k])]
    g["pcm_lengths"] = np.array([len(_PCM[short(f)]) for f in files + [query]], np.int64)
    g["pcm_crc"] = np.array([int(np.bitwise_xor.reduce(_PCM[short(f)].astype(np.int64) * (np.arange(len(_PCM[short(f)])) % 8191 + 1)))
                             for f in files + [query]], np.int64)
    for dens in DENSITIES:
        tag = "d%d" % int(dens)
        random.seed(2014)               # store()'s random.randint (no bucket fills here, but pin it)
        np.random.seed(2014)
        an = make_analyzer(dens, 1)
        ht = ref_ht.HashTable(hashbits=20, depth=100, maxtime=1 << 16)   # audfprint.py:421-436 defaults
        for k, f in enumerate(files):
            h = np.asarray(an.wavfile2hashes(short(f)), np.int32).reshape(-1, 2)
            g["%s/track%d/hashes" % (tag, k)] = h
            # `new` on 0*.mp3 then `add` on 1*.mp3 is one sequence of ingests (Makefile:27-29)
            dur, nh = an.ingest(ht, short(f))
            print(tag, short(f), "%.2f s" % dur, nh, "hashes")
        b = np.nonzero(ht.counts)[0]
        g[tag + "/db/params"] = np.array([20, 100, 16], np.int32)
        g[tag + "/db/buckets"] = b.astype(np.int32)
        g[tag + "/db/rows"] = ht.table[b]
        g[tag + "/db/counts"] = ht.counts[b]
        g[tag + "/db/hashesperid"] = np.asarray(ht.hashesperid, np.uint32)
        for shifts in (4, 1):           # 4 is what `match` uses (audfprint.py:295-297)
            qan = make_analyzer(dens, shifts)
            qh = np.asarray(qan.wavfile2hashes(short(query)), np.int32).reshape(-1, 2)
            g["%s/query_s%d/hashes" % (tag, shifts)] = qh
            for cfg, kw in MATCH_CONFIGS.items():
                mt = make_matcher(**kw)
                rows = mt.match_hashes(ht, qh)
                key = "%s/query_s%d/%s" % (tag, shifts, cfg)
                g[key + "/rows"] = np.asarray(rows, np.int64).reshape(-1, 7)
                msgs = mt.file_match_to_msgs(qan, ht, short(query))
                g[key + "/msgs"] = np.array(msgs)
                mt.verbose = False
                g[key + "/msgs_terse"] = np.array(mt.file_match_to_msgs(qan, ht, short(query)))
                print(key, rows[:2].tolist() if len(rows) else [], msgs[:1])
        # excerpts cut out of the committed tracks (5 s from 3 s in: not frame-aligned), matched
        # with 4 shifts like the command line does; tie flags from the reference's own hits
        for k in PCM_TRACKS:
            nm = "excerpt%d" % k
            _PCM[nm] = excerpt(_PCM[short(files[k])])
            qan = make_analyzer(dens, 4)
            qh = np.asarray(qan.wavfile2hashes(nm), np.int32).reshape(-1, 2)
            g["%s/%s/hashes" % (tag, nm)] = qh
            hits = np.asarray(ht.get_hits(qh))
            for cfg in ("top5", "exact_range_time", "tight"):
                mt = make_matcher(**MATCH_CONFIGS[cfg])
                rows = np.asarray(mt.match_hashes(ht, qh), np.int64).reshape(-1, 7)
                key = "%s/%s/%s" % (tag, nm, cfg)
                g[key + "/rows"] = rows
                g[key + "/ties"] = np.array(option_ties(hits, ht.hashesperid, rows, mt.threshcount, mt.search_depth))
                g[key + "/msgs"] = np.array(mt.file_match_to_msgs(qan, ht, nm))
                print(key, rows[:3].tolist(), g[key + "/ties"].tolist())
        # peak lists (the .afpk route, Makefile:50-56) of the query and one track
        pan = make_analyzer(dens, 1)
        for nm, src in (("query", short(query)), ("track4", short(files[4]))):
            pk = pan.wavfile2peaks(src)
            g["%s/%s/peaks" % (tag, nm)] = np.asarray(pk, np.int32).reshape(-1, 2)
    pcm_out = OUT.replace(".npz", "_pcm.npz")          # each file stays under 1 MB
    np.savez_compressed(pcm_out, **{k: v for k, v in g.items() if k.endswith("/pcm")})
    np.savez_compressed(OUT, **{k: v for k, v in g.items() if not k.endswith("/pcm")})
    for fn in (OUT, pcm_out):
        print("wrote", fn, os.path.getsize(fn), "bytes")


if __name__ == "__main__":
    main()
