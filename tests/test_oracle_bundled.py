"""CPU: the oracle against what the LIVE reference produced on its own bundled test
material (the reference's tests/data: Nine_Lives/*.mp3 and query.mp3, the files of the
reference's `make test`), stored in tests/golden/bundled.npz and bundled_pcm.npz by
oracle/make_golden_bundled.py.  The MP3s were decoded with FFmpeg's libraries at the
parameters of the reference's `ffmpeg -f s16le -ac 1 -ar 11025` pipe (oracle/ffdecode.py).

The first group runs anywhere (committed PCM of the query and of four tracks, reference
outputs for all thirteen).  The second group needs the reference's code and MP3s
(oracle/_ref/, made by build() from a reference checkout, or the checkout named by
$AFP_REFERENCE; it skips without them) and the vendored FFmpeg libraries: it re-decodes the
MP3s, checks the nine tracks whose PCM is not committed, and runs the UNMODIFIED reference
command line (`new`, `add`, `match`: Makefile:19-29) on the decoded audio to confirm the
stored report lines."""
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from oracle import afp_oracle as orc
from oracle import build_ref
from tests.conftest import expand_table, load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = build_ref.reference_dir() or ""
PCM_TRACKS = (0, 4, 8, 12)
DENSITIES = (100.0, 20.0)
# Matcher settings of oracle/make_golden_bundled.py on top of the command line's defaults
# (window 2, min-count 5, search-depth 100, time-quantile 0.05: audfprint.py:303-317,358-368)
CONFIGS = {
    "default": {},
    "top5": {},
    "exact": {"exact_count": True},
    "range": {"find_time_range": True},
    "exact_range_time": {"exact_count": True, "find_time_range": True},
    "tight": {"window": 1, "threshcount": 2, "search_depth": 4},
}


@pytest.fixture(scope="module")
def gb():
    return load_golden("bundled", "bundled_pcm")


def to_float(pcm):
    return pcm.astype(np.float32) / 32768.0


def excerpt(pcm):
    return pcm[3 * 11025:8 * 11025]


def oracle_rows(gb, tag, q, **kw):
    table, counts, hashbits, depth, mtb, hpi = expand_table(gb, tag + "/db")
    args = dict(window=2, threshcount=5, search_depth=100, quantile=0.05)
    args.update(kw)
    return orc.match_hashes(table, counts, hashbits, depth, mtb, hpi, q, **args)


@pytest.mark.parametrize("dens", DENSITIES)
def test_fingerprints_of_the_bundled_audio(gb, dens):
    tag = "d%d" % int(dens)
    q = to_float(gb["query/pcm"])
    assert np.array_equal(orc.fingerprint(q, density=dens, shifts=4), gb[tag + "/query_s4/hashes"])
    assert np.array_equal(orc.fingerprint(q, density=dens, shifts=1), gb[tag + "/query_s1/hashes"])
    assert np.array_equal(np.array(orc.find_peaks(q, density=dens), np.int32).reshape(-1, 2), gb[tag + "/query/peaks"])
    for k in PCM_TRACKS:
        d = to_float(gb["track%d/pcm" % k])
        assert np.array_equal(orc.fingerprint(d, density=dens), gb["%s/track%d/hashes" % (tag, k)]), k
        assert np.array_equal(orc.fingerprint(excerpt(d), density=dens, shifts=4), gb["%s/excerpt%d/hashes" % (tag, k)]), k
    pk = orc.find_peaks(to_float(gb["track4/pcm"]), density=dens)
    assert np.array_equal(np.array(pk, np.int32).reshape(-1, 2), gb[tag + "/track4/peaks"])


@pytest.mark.parametrize("dens", DENSITIES)
def test_database_of_the_thirteen_tracks(gb, dens):
    tag = "d%d" % int(dens)
    table, counts, hashbits, depth, mtb, hpi = expand_table(gb, tag + "/db")
    t = orc.Table(hashbits, depth, mtb)
    rng = random.Random(2014)
    for k, name in enumerate(gb["names"]):
        t.store(str(name), gb["%s/track%d/hashes" % (tag, k)], rng)
    assert np.array_equal(t.counts, counts) and np.array_equal(t.table, table)
    assert np.array_equal(t.hashesperid, hpi)


@pytest.mark.parametrize("dens", DENSITIES)
def test_match_rows_of_the_bundled_query_and_excerpts(gb, dens):
    tag = "d%d" % int(dens)
    nrows = 0
    for shifts in (4, 1):
        q = gb["%s/query_s%d/hashes" % (tag, shifts)]
        for cfg, kw in CONFIGS.items():
            want = gb["%s/query_s%d/%s/rows" % (tag, shifts, cfg)]
            got = oracle_rows(gb, tag, q, **kw)
            assert np.array_equal(got, want), (tag, shifts, cfg)
            nrows += len(want)
    for k in PCM_TRACKS:
        q = gb["%s/excerpt%d/hashes" % (tag, k)]
        for cfg in ("top5", "exact_range_time", "tight"):
            key = "%s/excerpt%d/%s" % (tag, k, cfg)
            want = gb[key + "/rows"]
            got = oracle_rows(gb, tag, q, **CONFIGS[cfg])
            tie_w, tie_c = gb[key + "/ties"]
            assert got.shape == want.shape and np.array_equal(got[:, 1], want[:, 1]), key
            assert int(want[0, 0]) == k and int(want[0, 2]) == 130          # 3 s = 129.2 hops, rounded by the shifts
            if not tie_w and not tie_c:
                assert np.array_equal(got, want), key
            elif not tie_w:
                assert sorted(map(tuple, got)) == sorted(map(tuple, want)), key
            nrows += len(want)
    assert nrows > 20


def test_bundled_query_is_found_in_full_circle(gb):
    """What the reference's README shows for `match query.mp3` (README.md:96-98): track 05."""
    for tag in ("d100", "d20"):
        rows = gb[tag + "/query_s4/default/rows"]
        assert len(rows) == 1 and str(gb["names"][rows[0, 0]]).endswith("05-Full_Circle.mp3")
        assert str(gb[tag + "/query_s4/default/msgs"][0]).startswith("Matched query.mp3 5.6 sec")


def test_mirror_report_lines_from_the_reference_rows(gb):
    """Host half of Matcher.file_match_to_msgs / match_file (sort_by_time, max_returns, the -R
    line, terse form) with the device calls replaced by the reference's own rows: the mirror
    prints the reference's lines (audfprint_match.py:354-420)."""
    from audfprint_b200 import Analyzer, Matcher
    overrides = {"default": {}, "top5": {"max_returns": 5}, "exact": {"max_returns": 5, "exact_count": True},
                 "range": {"max_returns": 5, "find_time_range": True},
                 "exact_range_time": {"max_returns": 5, "exact_count": True, "find_time_range": True,
                                      "sort_by_time": True},
                 "tight": {"max_returns": 3, "window": 1, "threshcount": 2, "search_depth": 4}}

    class Table(object):
        names = [str(n) for n in gb["names"]]
    checked = 0
    for tag in ("d100", "d20"):
        cases_ = [("query_s%d" % s, str(gb["query_name"]), cfg) for s in (4, 1) for cfg in overrides]
        cases_ += [("excerpt%d" % k, "excerpt%d" % k, cfg) for k in PCM_TRACKS for cfg in ("top5", "exact_range_time", "tight")]
        for qkey, qname, cfg in cases_:
            key = "%s/%s/%s" % (tag, qkey, cfg)
            if key + "/ties" in gb and any(gb[key + "/ties"]):
                continue
            mt = Matcher()
            mt.window, mt.threshcount, mt.max_returns, mt.search_depth = 2, 5, 1, 100
            mt.verbose, mt.time_quantile = True, 0.05
            for k, v in overrides[cfg].items():
                setattr(mt, k, v)
            an = Analyzer()
            an.wavfile2hashes = lambda fn, h=gb["%s/%s/hashes" % (tag, qkey)]: h
            mt.match_hashes = lambda ht, q, r=gb[key + "/rows"].astype(np.int32): r
            assert mt.file_match_to_msgs(an, Table, qname) == [str(x) for x in gb[key + "/msgs"]], key
            if key + "/msgs_terse" in gb:
                mt.verbose = False
                assert mt.file_match_to_msgs(an, Table, qname) == [str(x) for x in gb[key + "/msgs_terse"]], key
            checked += 1
    assert checked > 40


# ---- with the reference's code and MP3s only: the MP3s themselves and the live reference ------
def _have_decoder():
    try:
        from oracle import ffdecode
        ffdecode._load()
        return True
    except Exception:
        return False


live = pytest.mark.skipif(not (REF and os.path.isfile(os.path.join(REF, "tests", "data", "query.mp3")) and _have_decoder()),
                          reason="needs the reference checkout and the vendored FFmpeg libraries")


def _crc(pcm):
    return int(np.bitwise_xor.reduce(pcm.astype(np.int64) * (np.arange(len(pcm)) % 8191 + 1)))


@live
def test_decoding_is_reproducible_and_oracle_holds_on_all_thirteen(gb):
    from oracle import ffdecode
    data = os.path.join(REF, "tests", "data")
    names = [str(n) for n in gb["names"]] + [str(gb["query_name"])]
    for i, name in enumerate(names):
        pcm = ffdecode.decode(os.path.join(data, name))
        assert len(pcm) == gb["pcm_lengths"][i] and _crc(pcm) == gb["pcm_crc"][i], name
        if i in PCM_TRACKS:
            assert np.array_equal(pcm, gb["track%d/pcm" % i])
        if i < 13:
            for dens in DENSITIES:
                want = gb["d%d/track%d/hashes" % (int(dens), i)]
                assert np.array_equal(orc.fingerprint(to_float(pcm), density=dens), want), (name, dens)
    assert np.array_equal(ffdecode.decode(os.path.join(data, "query.mp3")), gb["query/pcm"])


CLI_DRIVER = r'''
import os, sys
ROOT, REF = sys.argv[1], sys.argv[2]
sys.path.insert(0, ROOT)
from tests.test_reference_cli_cpu import DRIVER
pre = DRIVER.split("sys.path.insert(0, REF)")[0]          # the docopt stand-in
sys.argv = [sys.argv[0], ROOT, REF, "ref", sys.argv[3]]
exec(pre)
sys.path.insert(0, REF)
import numpy as np
import audio_read
from oracle import ffdecode
audio_read.audio_read = ffdecode.audio_read               # where the ffmpeg pipe stands
import audfprint                                          # the reference's CLI, unmodified
for argv in argv_sets:
    audfprint.main(["audfprint"] + argv)
'''


@live
def test_reference_command_line_on_the_bundled_files(gb, tmp_path):
    """`make test_onecore` of the reference (Makefile:19-29) with the decoder in the place of
    the ffmpeg pipe: the report line is the one stored in the golden file."""
    data = os.path.join(REF, "tests", "data")
    db = str(tmp_path / "fpdbase.pklz")
    files = sorted(os.listdir(os.path.join(data, "Nine_Lives")))
    first = [os.path.join("Nine_Lives", f) for f in files if f.startswith("0")]
    rest = [os.path.join("Nine_Lives", f) for f in files if f.startswith("1")]
    text = ""
    for argv in (["new", "--dbase", db, "--density", "100"] + first,
                 ["add", "--dbase", db, "--density", "100"] + rest,
                 ["match", "--dbase", db, "--density", "100", "query.mp3"],
                 ["match", "--dbase", db, "--density", "100", "--find-time-range", "--exact-count",
                  "--max-matches", "5", "--sortbytime", "query.mp3"]):
        out = subprocess.run([sys.executable, "-c", CLI_DRIVER, ROOT, REF, repr([argv])],
                             capture_output=True, text=True, timeout=600, cwd=data)
        assert out.returncode == 0, out.stdout + out.stderr
        text += out.stdout
    lines = text.splitlines()
    assert str(gb["d100/query_s4/default/msgs"][0]) in lines
    assert str(gb["d100/query_s4/exact_range_time/msgs"][0]) in lines
    nh = int(np.sum(gb["d100/db/hashesperid"]))
    assert any(ln.startswith("Saved fprints for 13 files ( %d hashes)" % nh) for ln in lines)
