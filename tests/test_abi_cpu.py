"""CPU: the C-ABI library loads and exports every symbol include/afp.h declares;
host-side logic (packing, codecs, table bookkeeping) without any compute call."""
import os
import pickle
import random
import subprocess

import numpy as np
import pytest

import __graft_entry__ as entry
from audfprint_b200 import _lib, HashTable, Analyzer, Matcher
from audfprint_b200 import analyzer as an_mod
from oracle import afp_oracle as orc
from tests import cases
from tests.conftest import expand_table


@pytest.fixture(scope="module", autouse=True)
def built():
    entry.build()


def test_library_exports_every_declared_symbol():
    lib = _lib.load(check_symbols=True)
    syms = _lib.header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), s
    assert lib.afp_abi_version() == 2


def test_fft_index_algebra_host_check():
    out = subprocess.run([os.path.join(entry.ROOT, "build", "fft_host_check")], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_lib.AfpError):
        Analyzer().find_peaks(np.zeros(1000, np.float32), 11025)


@pytest.mark.parametrize("db", ["db", "db2"])
def test_store_matches_reference_table(golden_match, db):
    table, counts, hashbits, depth, mtb, hpi = expand_table(golden_match, db)
    random.seed(1234)
    ht = HashTable(hashbits=hashbits, depth=depth, maxtime=1 << mtb)
    for i in range(cases.DB_NTRACKS):
        ht.store("track%d" % i, golden_match["track%d/hashes" % i])
    assert np.array_equal(ht.counts, counts)
    assert np.array_equal(ht.table, table)
    assert np.array_equal(ht.hashesperid, hpi)
    assert ht.names[3] == "track3" and ht.dirty


def test_table_bookkeeping_roundtrip(tmp_path, golden_match):
    ht = HashTable(hashbits=12, depth=6, maxtime=1 << 10)
    random.seed(5)
    h0 = golden_match["track0/hashes"]
    h1 = golden_match["track1/hashes"]
    ht.store("a", h0)
    ht.store("b", h1)
    got = ht.retrieve("b")
    # retrieve returns what survived (bucket overflow drops some); all are real rows of b
    want = {(int(t) & 1023, int(h) & 4095) for t, h in h1}
    assert len(got) > 0 and {(int(t), int(h)) for t, h in got} <= want
    fn = str(tmp_path / "db.pklz")
    ht.save(fn)
    ht2 = HashTable(fn)
    assert np.array_equal(ht2.table, ht.table) and np.array_equal(ht2.counts, ht.counts)
    assert ht2.names == ["a", "b"] and not ht2.dirty
    ht2.remove("a")
    assert ht2.names[0] is None and ht2.hashesperid[0] == 0
    assert not np.any((ht2.table >> 10) == 1)
    with pytest.raises(ValueError):
        ht2.name_to_id("zzz")
    with pytest.raises(ValueError):
        HashTable(maxtime=1000)
    other = HashTable(hashbits=12, depth=6, maxtime=1 << 10)
    other.store("c", h0[:50])
    n_before = len(ht2.names)
    ht2.merge(other)
    assert ht2.names[n_before] == "c"
    p = pickle.loads(pickle.dumps(ht))
    assert np.array_equal(p.table, ht.table)


def test_codecs_are_byte_compatible(tmp_path):
    rows = [(0, 5), (3, 1048575), (70000, 12)]
    fn = str(tmp_path / "x.afpt")
    an_mod.hashes_save(fn, rows)
    raw = open(fn, "rb").read()
    assert raw[:16] == b"audfprinthashV00" and len(raw) == 16 + 8 * 3
    assert an_mod.hashes_load(fn) == rows
    fk = str(tmp_path / "x.afpk")
    an_mod.peaks_save(fk, rows)
    assert open(fk, "rb").read()[:16] == b"audfprintpeakV00"
    assert an_mod.peaks_load(fk) == rows
    with pytest.raises(IOError):
        an_mod.hashes_load(fk)


def test_hash_packing_matches_oracle():
    lms = [(5, 10, 40, 2), (7, 255, 225, 62), (9, 0, 30, 33)]
    assert np.array_equal(an_mod.landmarks2hashes(lms), orc.landmarks_to_hashes(lms))
    assert an_mod.hashes2landmarks(an_mod.landmarks2hashes(lms)) == lms
    assert an_mod.landmarks2hashes([]).shape == (0, 2)


def test_objects_pickle_without_device_state():
    a = pickle.loads(pickle.dumps(Analyzer(density=70.0)))
    assert a.density == 70.0 and a.shifts == 1 and a.maxpksperframe == 5
    m = pickle.loads(pickle.dumps(Matcher()))
    assert m.window == 1 and m.threshcount == 5
    m.illustrate = True
    with pytest.raises(NotImplementedError):
        m._params()


def test_loads_database_pickled_by_the_reference():
    """tests/golden/ref_db.pklz was written by the live reference's HashTable.save."""
    import os
    from tests.conftest import GOLDEN
    ht = HashTable(os.path.join(GOLDEN, "ref_db.pklz"))
    want = np.load(os.path.join(GOLDEN, "ref_db_arrays.npz"))
    assert np.array_equal(ht.table, want["table"]) and np.array_equal(ht.counts, want["counts"])
    assert np.array_equal(ht.hashesperid, want["hashesperid"])
    assert ht.names == ["ref_track%d" % i for i in range(6)]
    assert (ht.hashbits, ht.depth, ht.maxtimebits) == (10, 4, 10) and ht.params["samplerate"] == 11025


def test_saved_database_has_the_reference_class_path(tmp_path):
    import gzip
    import pickletools
    ht = HashTable(hashbits=8, depth=3, maxtime=1 << 8)
    ht.store("x", [(1, 5), (2, 5), (3, 77)])
    fn = str(tmp_path / "db.pklz")
    ht.save(fn, params={"k": 1})
    ops = [(op.name, arg) for op, arg, _ in pickletools.genops(gzip.open(fn, "rb").read())]
    strings = [a for _, a in ops if isinstance(a, str)]
    assert "hash_table" in strings and "HashTable" in strings
    assert not any("audfprint_b200" in a for a in strings)
    ht2 = HashTable(fn)
    assert np.array_equal(ht2.table, ht.table) and ht2.params == {"k": 1} and ht2.names == ["x"]
    from oracle import build_ref
    ref = build_ref.reference_dir()
    if ref:                                      # with the reference's code at hand: it reads our file
        import subprocess
        import sys
        code = ("import sys; sys.path.insert(0, %r); import hash_table as h; t = h.HashTable(%r); "
                "print(t.names, int(t.counts.sum()), t.get_hits([[0, 5]]).tolist())" % (ref, fn))
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        assert "['x'] 3 [[0, 1, 5, 0], [0, 2, 5, 0]]" in out.stdout


@pytest.mark.parametrize("db", ["db", "db2"])
def test_matcher_option_postprocessing_host_logic(golden_match, golden_options, db, monkeypatch):
    """Matcher's exact_count / find_time_range / hashesfor host stage, fed with the reference's
    own hits and the oracle's candidate list in place of the two device calls (those are
    checked on the GPU in test_gpu_parity.py)."""
    from oracle import afp_oracle as orc
    from tests.conftest import expand_table, option_ties
    gm, go = golden_match, golden_options
    table, counts, hashbits, depth, mtb, hpi = expand_table(gm, db)
    nexact = 0
    for j in range(cases.DB_QUERIES):
        for tag in ("clean", "noisy"):
            key = "q%d_%s" % (j, tag)
            q = gm[key + "/q"]
            hits = gm["%s/%s/hits" % (db, key)]
            for cfg in ("tr", "ex", "extr", "trb"):
                exact, trange, window, thresh, sdepth = (int(x) for x in go["cfg_" + cfg])
                m = Matcher()
                m.window, m.threshcount, m.search_depth = window, thresh, sdepth
                m.exact_count, m.find_time_range = bool(exact), bool(trange)
                ids, raws = orc.rank_candidates(hits, hpi, thresh, sdepth)
                approx = orc.offset_histogram_rows(hits, ids, raws, window, thresh)
                monkeypatch.setattr(m, "_device_rows_and_candidates", lambda ht, q_: (approx, ids, raws))

                class _HT:                       # stands in for the device probe
                    def get_hits(self, q_):
                        return hits
                want = go["%s/%s/rows_%s" % (db, key, cfg)]
                tie_w, tie_c = option_ties(hits, hpi, want, thresh, sdepth)
                if len(want) and not tie_w and not tie_c:
                    rows, pairs = m.match_hashes(_HT(), q, hashesfor=0)
                    assert np.array_equal(rows, want), (db, key, cfg)
                    assert np.array_equal(pairs, go["%s/%s/pairs_%s" % (db, key, cfg)])
                    nexact += 1
                else:
                    rows = m.match_batch(_HT(), [q])[0]
                    assert rows.shape == want.shape and np.array_equal(rows[:, 1], want[:, 1])
    assert nexact > 15


def test_table_bookkeeping_equals_the_reference(golden_match, capsys):
    """store / merge (np.random reservoir) / remove / id-slot reuse / retrieve / list: the mirror
    class replays the scripted sequence of oracle/make_golden_table_ops.py and must reproduce the
    live reference's table after every step."""
    from oracle.make_golden_table_ops_replay import run
    from tests.conftest import GOLDEN
    want = np.load(os.path.join(GOLDEN, "table_ops.npz"))
    seen = []

    def record(tag, ht):
        seen.append(tag)
        assert np.array_equal(ht.table, want[tag + "/table"]), tag
        assert np.array_equal(ht.counts, want[tag + "/counts"]), tag
        assert np.array_equal(ht.hashesperid, want[tag + "/hashesperid"]), tag
        assert ["" if n is None else n for n in ht.names] == want[tag + "/names"].tolist(), tag
    ht, r9, rlate, lines = run(HashTable, golden_match, record)
    assert seen == ["a", "b", "merged", "removed", "reused"]
    assert np.array_equal(r9, want["retrieve_track9"]) and r9.dtype == np.int32
    assert np.array_equal(rlate, want["retrieve_late"])
    assert lines == want["list_lines"].tolist()
    assert ht.names[3] == "late" and "Removed track3 ( 335 hashes)." in capsys.readouterr().out


def test_loads_matlab_database_like_the_reference():
    """tests/golden/matlab_db.mat (oracle/make_golden_mat.py) -> the attributes the live reference's
    loader produced for the same file."""
    from tests.conftest import GOLDEN
    ht = HashTable(os.path.join(GOLDEN, "matlab_db.mat"))
    want = np.load(os.path.join(GOLDEN, "matlab_db_arrays.npz"))
    assert np.array_equal(ht.table, want["table"]) and np.array_equal(ht.counts, want["counts"])
    assert np.array_equal(ht.hashesperid, want["hashesperid"])
    assert [n if isinstance(n, str) else "" for n in ht.names] == want["names"].tolist()
    assert [ht.hashbits, ht.depth, ht.maxtimebits] == want["geometry"].tolist() and isinstance(ht.depth, int)
    got = [ht.params[k] for k in ("mat_version", "hoptime", "targetsr", "nojenkins")]
    assert np.allclose(got, want["params"]) and not ht.dirty
    assert ht.table.dtype == np.uint32 and ht.table.flags["C_CONTIGUOUS"] and ht.counts.dtype == np.int32


def test_get_entry_reads_one_bucket(golden_match):
    table, counts, hashbits, depth, mtb, hpi = expand_table(golden_match, "db2")
    ht = HashTable(hashbits=hashbits, depth=depth, maxtime=1 << mtb)
    ht.table, ht.counts, ht.hashesperid = table, counts, hpi
    b = int(np.argmax(counts))                       # an over-full bucket: only `depth` entries exist
    got = ht.get_entry(b)
    assert got.shape == (depth, 2) and got.dtype == np.int32
    hits = orc.get_hits(table, counts, hashbits, depth, mtb, np.array([[0, b]], np.int32))
    assert np.array_equal(got, hits[:, :2])          # query time 0: dtime == stored time
    assert ht.get_entry(int(np.argmin(counts))).shape == (int(counts.min()), 2)
