"""GPU: the CUDA path on the reference's OWN bundled test material (the Nine_Lives excerpts
and query.mp3 of the reference's tests/data - what `make test` of the reference runs,
Makefile:12-29), against what the LIVE reference produced on the same decoded PCM
(tests/golden/bundled.npz and bundled_pcm.npz, oracle/make_golden_bundled.py).
BASELINE.json north_star: "match results bit-identical to the reference on the bundled tests/data queries".

Real, heavily clipped music instead of the synthetic tracks of the other tests; hashes, peaks,
table arrays, match rows and report lines are compared bit for bit.  (The file sorts last so
that the synthetic-input suite reports first.)"""
import random

import numpy as np
import pytest

from audfprint_b200 import Analyzer, HashTable, Matcher
from oracle import afp_oracle as orc
from tests.conftest import expand_table, load_golden

pytestmark = pytest.mark.gpu
PCM_TRACKS = (0, 4, 8, 12)
DENSITIES = (100.0, 20.0)
MATCH_CONFIGS = {           # oracle/make_golden_bundled.py
    "default": {},
    "top5": {"max_returns": 5},
    "exact": {"max_returns": 5, "exact_count": True},
    "range": {"max_returns": 5, "find_time_range": True},
    "exact_range_time": {"max_returns": 5, "exact_count": True, "find_time_range": True, "sort_by_time": True},
    "tight": {"max_returns": 3, "window": 1, "threshcount": 2, "search_depth": 4},
}


@pytest.fixture(scope="module")
def gb():
    return load_golden("bundled", "bundled_pcm")


@pytest.fixture(scope="module")
def pcm(gb):
    """name -> int16 PCM, under the names the reference saw."""
    out = {str(gb["query_name"]): gb["query/pcm"]}
    for k in PCM_TRACKS:
        out[str(gb["names"][k])] = gb["track%d/pcm" % k]
        out["excerpt%d" % k] = gb["track%d/pcm" % k][3 * 11025:8 * 11025].copy()
    return out


def make_analyzer(pcm, density, shifts):
    """audfprint.py:280-299 with the command line's defaults; the reader hands out the decoded
    PCM exactly as the reference's reader does (float32 / 32768, audio_read.py:102-116)."""
    an = Analyzer()
    an.density = density
    an.shifts = shifts
    an.reader = lambda fn, sr=None, channels=None: (pcm[fn].astype(np.float32) / 32768.0, 11025)
    return an


def make_matcher(**kw):
    """audfprint.py:303-317 with the command line's defaults, then the overrides."""
    mt = Matcher()
    mt.window, mt.threshcount, mt.max_returns, mt.search_depth = 2, 5, 1, 100
    mt.verbose = True
    mt.time_quantile = 0.05
    for k, v in kw.items():
        setattr(mt, k, v)
    return mt


def golden_table(gb, tag):
    table, counts, hashbits, depth, mtb, hpi = expand_table(gb, tag + "/db")
    ht = HashTable(hashbits=hashbits, depth=depth, maxtime=1 << mtb)
    ht.table, ht.counts, ht.hashesperid = table, counts, hpi
    ht.names = [str(n) for n in gb["names"]]
    return ht


def rows2(x):
    return np.asarray(x, np.int32).reshape(-1, 2)


@pytest.mark.parametrize("dens", DENSITIES)
def test_fingerprints_of_the_bundled_audio(gb, pcm, dens):
    tag = "d%d" % int(dens)
    qn = str(gb["query_name"])
    for shifts in (4, 1):
        an = make_analyzer(pcm, dens, shifts)
        want = gb["%s/query_s%d/hashes" % (tag, shifts)]
        assert np.array_equal(rows2(an.wavfile2hashes(qn)), want)                  # float32 through the reader
        assert np.array_equal(an.fingerprint_batch([pcm[qn]])[0], want)            # int16 straight in
        assert np.array_equal(want, orc.fingerprint(pcm[qn].astype(np.float32) / 32768.0, density=dens, shifts=shifts))
    an = make_analyzer(pcm, dens, 1)
    names = [str(gb["names"][k]) for k in PCM_TRACKS]
    got = an.fingerprint_batch([pcm[n] for n in names])                            # one ragged device call
    for k, n, h in zip(PCM_TRACKS, names, got):
        assert np.array_equal(h, gb["%s/track%d/hashes" % (tag, k)]), n
        assert np.array_equal(rows2(an.wavfile2hashes(n)), gb["%s/track%d/hashes" % (tag, k)]), n
    an4 = make_analyzer(pcm, dens, 4)
    got = an4.fingerprint_batch([pcm["excerpt%d" % k] for k in PCM_TRACKS])
    for k, h in zip(PCM_TRACKS, got):
        assert np.array_equal(h, gb["%s/excerpt%d/hashes" % (tag, k)]), k
    # peak lists (the --precompute-peaks route, audfprint_analyze.py:345-383)
    assert np.array_equal(rows2(an.wavfile2peaks(qn)), gb[tag + "/query/peaks"])
    assert np.array_equal(rows2(an.wavfile2peaks(str(gb["names"][4]))), gb[tag + "/track4/peaks"])


@pytest.mark.parametrize("dens", DENSITIES)
def test_database_of_the_thirteen_tracks(gb, pcm, dens):
    """`new` + `add` of the Makefile: per-track store() of the reference's hashes gives the
    reference's table; the device-side batched ingest of the four committed tracks gives the
    table the oracle builds from the reference's hashes of those tracks."""
    tag = "d%d" % int(dens)
    want = golden_table(gb, tag)
    random.seed(2014)
    ht = HashTable(hashbits=20, depth=100, maxtime=1 << 16)
    for k, name in enumerate(gb["names"]):
        ht.store(str(name), gb["%s/track%d/hashes" % (tag, k)])
    assert np.array_equal(ht.counts, want.counts) and np.array_equal(ht.table, want.table)
    assert np.array_equal(np.asarray(ht.hashesperid), np.asarray(want.hashesperid))
    assert ht.names == want.names
    names = [str(gb["names"][k]) for k in PCM_TRACKS]
    random.seed(2014)
    dev = HashTable(hashbits=20, depth=100, maxtime=1 << 16)
    counts = make_analyzer(pcm, dens, 1).ingest_batch(dev, names, [pcm[n] for n in names])
    t = orc.Table(20, 100, 16)
    rng = random.Random(2014)
    for k, n in zip(PCM_TRACKS, names):
        t.store(n, gb["%s/track%d/hashes" % (tag, k)], rng)
    assert counts == [int(x) for x in t.hashesperid]
    assert np.array_equal(dev.counts, t.counts) and np.array_equal(dev.table, t.table)
    assert dev.names == names


@pytest.mark.parametrize("dens", DENSITIES)
def test_match_of_the_bundled_query(gb, pcm, dens):
    """`audfprint match --dbase fpdbase.pklz query.mp3` (Makefile:19-20): rows and report lines."""
    tag = "d%d" % int(dens)
    ht = golden_table(gb, tag)
    qn = str(gb["query_name"])
    for shifts in (4, 1):
        qan = make_analyzer(pcm, dens, shifts)
        q = gb["%s/query_s%d/hashes" % (tag, shifts)]
        for cfg, kw in MATCH_CONFIGS.items():
            key = "%s/query_s%d/%s" % (tag, shifts, cfg)
            mt = make_matcher(**kw)
            assert np.array_equal(mt.match_hashes(ht, q), gb[key + "/rows"]), key
            assert mt.file_match_to_msgs(qan, ht, qn) == [str(s) for s in gb[key + "/msgs"]], key
            mt.verbose = False
            assert mt.file_match_to_msgs(qan, ht, qn) == [str(s) for s in gb[key + "/msgs_terse"]], key
    # hits of the query rows, against the oracle's restatement of get_hits on the same table
    q = gb[tag + "/query_s4/hashes"]
    want_hits = orc.get_hits(ht.table, ht.counts, 20, 100, 16, q)
    assert np.array_equal(ht.get_hits(q), want_hits) and len(want_hits) > 10


@pytest.mark.parametrize("dens", DENSITIES)
def test_match_of_excerpts_cut_from_the_tracks(gb, pcm, dens):
    tag = "d%d" % int(dens)
    ht = golden_table(gb, tag)
    nexact = 0
    for cfg in ("top5", "exact_range_time", "tight"):
        mt = make_matcher(**MATCH_CONFIGS[cfg])
        qan = make_analyzer(pcm, dens, 4)
        qs = [gb["%s/excerpt%d/hashes" % (tag, k)] for k in PCM_TRACKS]
        batch = mt.match_batch(ht, qs)                                   # all four in one device call
        for k, q, brows in zip(PCM_TRACKS, qs, batch):
            key = "%s/excerpt%d/%s" % (tag, k, cfg)
            want = gb[key + "/rows"]
            tie_w, tie_c = gb[key + "/ties"]
            rows = mt.match_hashes(ht, q)
            assert rows.shape == want.shape and np.array_equal(rows[:, 1], want[:, 1]), key
            assert rows[0, 0] == k and rows[0, 2] == 130
            assert sorted(map(tuple, brows)) == sorted(map(tuple, rows)), key
            if not tie_w and not tie_c:
                assert np.array_equal(rows, want), key
                assert mt.file_match_to_msgs(qan, ht, "excerpt%d" % k) == [str(s) for s in gb[key + "/msgs"]], key
                nexact += 1
            elif not tie_w:
                assert sorted(map(tuple, rows)) == sorted(map(tuple, want)), key
    assert nexact >= 8
