"""Host-side behaviour of the API mirror that needs no GPU: report strings, pickling
hygiene, device-copy bookkeeping."""
import gzip
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

from audfprint_b200 import Analyzer, HashTable, Matcher
from oracle import build_ref
from tests import cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = build_ref.reference_dir() or ""          # the reference's code, if it is at hand

# What the live reference's Matcher.file_match_to_msgs returns (audfprint_match.py:381-420) when
# match_file yields these rows; generated in the build container by patching match_file on the
# reference class (the strings are its output, not code).
ROWS = np.array([[1, 123, -45, 200, 0, 17, 402], [2, 9, 1033, 40, 3, 0, 12]], np.int32)
NAMES = ["a.mp3", "dir/b song.wav", "c"]
QRY = "query file.mp3"
GOLDEN_MSGS = {
    (0, 0, 1): ['query file.mp3\tdir/b song.wav', 'query file.mp3\tc'],
    (0, 0, 0): ['query file.mp3\t'],
    (0, 1, 1): ['query file.mp3\tdir/b song.wav', 'query file.mp3\tc'],
    (0, 1, 0): ['query file.mp3\t'],
    (1, 0, 1): ['Matched query file.mp3 12.3 sec 567 raw hashes as dir/b song.wav at   -1.0 s with   123 of   200 '
                'common hashes at rank  0',
                'Matched query file.mp3 12.3 sec 567 raw hashes as c at   24.0 s with     9 of    40 common hashes '
                'at rank  3'],
    (1, 0, 0): ['NOMATCH query file.mp3 12.3 sec 567 raw hashes'],
    (1, 1, 1): ['Matched    8.9 s starting at    0.4 s in query file.mp3 to time   -0.7 s in dir/b song.wav with   '
                '123 of   200 common hashes at rank  0',
                'Matched    0.3 s starting at    0.0 s in query file.mp3 to time   24.0 s in c with     9 of    40 '
                'common hashes at rank  3'],
    (1, 1, 0): ['NOMATCH query file.mp3 12.3 sec 567 raw hashes'],
}


class _Names:
    names = NAMES


def test_report_lines_equal_the_reference_including_time_range_branch():
    for (verbose, ftr, hit), want in GOLDEN_MSGS.items():
        m = Matcher()
        m.verbose, m.find_time_range = bool(verbose), bool(ftr)
        rows = ROWS if hit else ROWS[:0]
        m.match_file = lambda an, ht, q, number=None, rows=rows: (rows, 12.34, 567)
        assert m.file_match_to_msgs(Analyzer(), _Names(), QRY) == want, (verbose, ftr, hit)


def test_save_leaves_no_stand_in_module_behind(tmp_path):
    """ADVICE r1: HashTable.save registered a stub `hash_table` module and never removed it."""
    code = r"""
import sys, os
sys.path.insert(0, %r)
from audfprint_b200 import HashTable
ht = HashTable(hashbits=8, depth=4, maxtime=256)
ht.store("x", [(1, 2), (3, 4)])
assert "hash_table" not in sys.modules
ht.save(%r)
assert "hash_table" not in sys.modules, "stand-in module leaked"
if os.path.isdir(%r):
    sys.path.insert(0, %r)
    import hash_table                      # the REAL reference module, usable after our save
    ref = hash_table.HashTable(%r)
    assert ref.names == ["x"] and int(ref.counts.sum()) == 2
    ht.save(%r)                            # with the real module loaded the real class is used
    assert sys.modules["hash_table"] is hash_table
print("ok")
""" % (ROOT, str(tmp_path / "a.pklz"), REF, REF, str(tmp_path / "a.pklz"), str(tmp_path / "b.pklz"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stdout + out.stderr
    with gzip.open(tmp_path / "a.pklz", "rb") as f:
        assert b"hash_table" in f.read(4096)


def test_device_stamp_is_unique_per_table_and_tracks_rebinding():
    """ADVICE r1: the freshness stamp must not be reusable by another table, and rebinding the
    public arrays must change it."""
    stamps = set()
    for _ in range(50):
        ht = HashTable(hashbits=6, depth=2, maxtime=64)
        stamps.add(ht._stamp())
        del ht
    assert len(stamps) == 50
    ht = HashTable(hashbits=6, depth=2, maxtime=64)
    s0 = ht._stamp()
    ht.table = np.zeros((64, 2), np.uint32)
    s1 = ht._stamp()
    ht.counts = np.zeros(64, np.int32)
    s2 = ht._stamp()
    ht.depth = 2
    ht.store("a", [(0, 1)])
    s3 = ht._stamp()
    ht.table[0, 0] = 7
    ht.touch()
    s4 = ht._stamp()
    assert len({s0, s1, s2, s3, s4}) == 5
    clone = pickle.loads(pickle.dumps(ht))
    assert clone._stamp()[0] != ht._stamp()[0]
    assert np.array_equal(clone.table, ht.table) and clone.names == ht.names
    assert "table" in ht.__getstate__() and "_table" not in ht.__getstate__()


# ---- Matcher options: the vectorised batch finish against the per-query one --------------------
def _emulated_device_results(table, counts, hashbits, depth, mtb, hpi, queries, window, thresh, sdepth, maxalign=100):
    """What the two device calls of Matcher.match_batch hand to the host finish (hits of every
    query row; publish-mode candidate lists and approximate rows, ranks past maxdepth included),
    computed with the oracle."""
    from oracle import afp_oracle as orc
    hits_l, rows_l, cand, cnts = [], [], np.zeros((len(queries), max(sdepth, 1), 3)), np.zeros((len(queries), 2), np.int32)
    for i, q in enumerate(queries):
        h = orc.get_hits(table, counts, hashbits, depth, mtb, q)
        hits_l.append(h)
        if len(h) == 0:
            rows_l.append(np.zeros((0, 7), np.int32))
            continue
        ids, raw = np.unique(h[:, 0], return_counts=True)
        wtd = raw / hpi[ids].astype(float)
        order = np.lexsort((-ids, -wtd))[:sdepth]                      # weight desc, id desc
        cnts[i] = (len(order), int(np.count_nonzero(raw > thresh)))
        cand[i, :len(order)] = np.stack([ids[order], raw[order], wtd[order]], axis=1)
        rows_l.append(orc.offset_histogram_rows(h, ids[order], raw[order], window, thresh, maxalign))
    hoff = np.concatenate([[0], np.cumsum([len(h) for h in hits_l])]).astype(np.int64)
    roff = np.concatenate([[0], np.cumsum([len(r) for r in rows_l])]).astype(np.int64)
    return (np.concatenate(hits_l) if hits_l else np.zeros((0, 4), np.int32), hoff,
            np.concatenate(rows_l) if rows_l else np.zeros((0, 7), np.int32), roff, cand, cnts)


@pytest.mark.parametrize("db", ["db", "db2"])
def test_options_batch_finish_equals_the_per_query_finish(golden_match, golden_options, db):
    """Matcher._finish_options_batch (array operations over the whole batch) returns the rows of
    Matcher._match_with_options query by query - which the GPU tests pin to the live reference -
    for every flag combination, incl. empty queries and candidate lists cut by search_depth."""
    from audfprint_b200 import Matcher
    from tests.conftest import expand_table
    gm = golden_match
    table, counts, hashbits, depth, mtb, hpi = expand_table(gm, db)
    qs = [gm["q%d_%s/q" % (j, tag)] for j in range(cases.DB_QUERIES) for tag in ("clean", "noisy")]
    qs.insert(3, np.zeros((0, 2), np.int32))
    qs.append(np.concatenate([qs[0], qs[5]]))                      # two tracks in one query
    nrows = 0
    for exact, trange, window, thresh, sdepth, quant in [(True, False, 2, 5, 100, 0.02), (False, True, 2, 5, 100, 0.05),
                                                         (True, True, 1, 3, 10, 0.02), (False, True, 1, 2, 3, 0.3),
                                                         (True, True, 0, 1, 4, 0.5), (True, False, 3, 2, 1, 0.02)]:
        m = Matcher()
        m.window, m.threshcount, m.search_depth, m.time_quantile = window, thresh, sdepth, quant
        m.exact_count, m.find_time_range = exact, trange
        hits, hoff, rows, roff, cand, cnts = _emulated_device_results(table, counts, hashbits, depth, mtb, hpi, qs,
                                                                      window, thresh, sdepth)
        got, goff = m._finish_options_batch(hits, hoff, rows, roff, cand, cnts)
        assert got.dtype == np.int32 and goff[-1] == len(got)
        for i, q in enumerate(qs):
            pre = (hits[hoff[i]:hoff[i + 1]], rows[roff[i]:roff[i + 1]], cand[i], cnts[i])
            want = m._match_with_options(None, q, device_results=pre)
            assert np.array_equal(got[goff[i]:goff[i + 1]], want), (db, exact, trange, window, thresh, sdepth, i)
            nrows += len(want)
        # the reference's rows where the golden file has this configuration (tie-free cases)
    assert nrows > 300


def test_options_batch_finish_keeps_the_reference_pair_packing_quirk():
    """encpowerof2(max query time) is one bit short when that time is a power of two
    (audfprint_match.py:46-48,157): (t = 2^k, hash h) and (t = 0, hash h + 1) then pack to the same
    key and count once in the reference.  Both finishes reproduce that."""
    from audfprint_b200 import Matcher
    # one track (id 0), offset 5: hits [id, dtime, hash, qtime]
    hits = np.array([[0, 5, 7, 8], [0, 5, 8, 0], [0, 5, 9, 3], [0, 5, 10, 4], [0, 5, 11, 5]], np.int32)
    hoff = np.array([0, 5], np.int64)
    cand = np.zeros((1, 4, 3)); cand[0, 0] = (0, 5, 1.0)
    cnts = np.array([[1, 1]], np.int32)
    rows = np.array([[0, 5, 5, 5, 0, 0, 0]], np.int32)
    m = Matcher()
    m.window, m.threshcount, m.search_depth, m.exact_count = 1, 2, 4, True
    got, goff = m._finish_options_batch(hits, hoff, rows, np.array([0, 1], np.int64), cand, cnts)
    want = m._match_with_options(None, np.zeros((5, 2), np.int32), device_results=(hits, rows, cand[0], cnts[0]))
    assert np.array_equal(got, want) and got[0, 1] == 4          # 5 hits, 4 distinct packed keys


def test_options_batch_finish_fuzz():
    """Random hit lists with few ids and offsets (adjacent histogram bins, overlapping windows,
    several alignments per id, largest query times that are powers of two, quantiles 0 and 0.5,
    empty queries): the batch finish equals the per-query finish row for row."""
    rng = np.random.default_rng(7)
    checked = 0
    for trial in range(80):
        nq, sd = int(rng.integers(1, 6)), int(rng.integers(1, 8))
        thresh, window = int(rng.integers(1, 5)), int(rng.integers(0, 4))
        hits_l, rows_l, cand, cnts = [], [], np.zeros((nq, sd, 3)), np.zeros((nq, 2), np.int32)
        for i in range(nq):
            n = int(rng.integers(0, 120))
            maxq = int(rng.choice([8, 16, 64, 100, 37]))
            h = np.stack([rng.integers(0, 6, n), rng.integers(-6, 7, n), rng.integers(0, 12, n),
                          rng.integers(0, maxq + 1, n)], axis=1).astype(np.int32)
            hits_l.append(h)
            rr = []
            if n:
                ids, raw = np.unique(h[:, 0], return_counts=True)
                w = raw / rng.integers(1, 50, len(ids))
                o = np.lexsort((-ids, -w))[:sd]
                cnts[i] = (len(o), int(np.count_nonzero(raw > thresh)))
                cand[i, :len(o)] = np.stack([ids[o], raw[o], w[o]], axis=1)
                for rank, (id_, r_) in enumerate(zip(ids[o], raw[o])):        # rows at offsets that have hits
                    dts = np.unique(h[h[:, 0] == id_, 1])
                    for md in rng.choice(dts, size=min(len(dts), int(rng.integers(0, 3))), replace=False):
                        rr.append([id_, 5, md, r_, rank, 0, 0])
            rows_l.append(np.array(rr, np.int32).reshape(-1, 7))
        hoff = np.concatenate([[0], np.cumsum([len(h) for h in hits_l])]).astype(np.int64)
        roff = np.concatenate([[0], np.cumsum([len(r) for r in rows_l])]).astype(np.int64)
        hits, rows = np.concatenate(hits_l), np.concatenate(rows_l)
        for exact, trange in [(True, False), (True, True), (False, True)]:
            m = Matcher()
            m.window, m.threshcount, m.search_depth, m.exact_count, m.find_time_range = window, thresh, sd, exact, trange
            m.time_quantile = float(rng.choice([0.02, 0.05, 0.3, 0.5, 0.0]))
            got, goff = m._finish_options_batch(hits, hoff, rows, roff, cand, cnts)
            for i in range(nq):
                pre = (hits[hoff[i]:hoff[i + 1]], rows[roff[i]:roff[i + 1]], cand[i], cnts[i])
                want = m._match_with_options(None, np.zeros((1, 2), np.int32), device_results=pre)
                assert np.array_equal(got[goff[i]:goff[i + 1]], want), (trial, exact, trange, i)
                checked += 1
    assert checked > 500
