"""INTEGRATION.md option A, executed: the UNMODIFIED reference command line (audfprint.py) with
the three import swaps - `audfprint_analyze`, `audfprint_match`, `hash_table` resolving to
audfprint_b200's mirrors - run on precomputed .afpt inputs (host-only path: no GPU needed), and
compared with the same commands run on the pure reference.  `match` needs the device and is
covered by the GPU tests through the same classes.

The reference's code comes from oracle/_ref/, which build() compiles from a reference checkout, or
from the checkout named by $AFP_REFERENCE; the tests skip where neither is present.
docopt is not installed in the image; a small stand-in parses the reference's own USAGE text."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import build_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = build_ref.reference_dir()

pytestmark = pytest.mark.skipif(REF is None,
                                reason="reference checkout not present")

DRIVER = r'''
import os, re, sys, types
ROOT, REF, swap = sys.argv[1], sys.argv[2], sys.argv[3] == "swap"
argv_sets = eval(sys.argv[4])
sys.path.insert(0, ROOT)

def mini_docopt(usage, version=None, argv=None):
    """Just enough of docopt for the reference's USAGE: commands, `--opt <val>` with
    [default: x], flags, positional <file>..."""
    opts, short = {}, {}
    for line in usage.split("Options:")[1].splitlines():
        m = re.match(r"\s+(?:(-\w)(?: <\w+>)?, )?(--[\w-]+)( <\w+>)?\s+(.*)", line)
        if not m:
            continue
        s, name, arg, rest = m.groups()
        takes = bool(arg) or (s is not None and re.search(re.escape(s) + r" <", line) is not None)
        d = re.search(r"\[default: (.*)\]", rest)
        opts[name] = (takes, (d.group(1) if d else None) if takes else False)
        if s:
            short[s] = name
    cmds = re.search(r"Usage: audfprint \(([^)]*)\)", usage).group(1).replace(" ", "").split("|")
    out = {c: False for c in cmds}
    out.update({k: v[1] for k, v in opts.items()})
    out["<file>"] = []
    it = iter(argv)
    for a in it:
        a = short.get(a, a)
        if a in cmds:
            out[a] = True
        elif a in opts:
            out[a] = next(it) if opts[a][0] else True
        else:
            out["<file>"].append(a)
    return out

mod = types.ModuleType("docopt")
mod.docopt = mini_docopt
sys.modules["docopt"] = mod
if swap:
    # the three import swaps of INTEGRATION.md, option A
    import audfprint_b200.analyzer, audfprint_b200.matcher, audfprint_b200.hash_table
    sys.modules["audfprint_analyze"] = audfprint_b200.analyzer
    sys.modules["audfprint_match"] = audfprint_b200.matcher
    sys.modules["hash_table"] = audfprint_b200.hash_table
sys.path.insert(0, REF)
import random
import numpy as np
import audfprint                      # the reference's CLI module, unmodified
for argv in argv_sets:
    random.seed(2024)
    np.random.seed(2024)
    audfprint.main(["audfprint"] + argv)
'''


def _run(tmp, swap, argv_sets):
    """One process per command, as the command line is used (the reference's save() leaves the
    closing of its gzip stream to interpreter exit)."""
    text = ""
    for argv in argv_sets:
        out = subprocess.run([sys.executable, "-c", DRIVER, ROOT, REF, "swap" if swap else "ref", repr([argv])],
                             capture_output=True, text=True, timeout=600, cwd=tmp)
        assert out.returncode == 0, out.stdout + out.stderr
        text += out.stdout
    return text


def _load_db(path):
    sys.path.insert(0, ROOT)
    from audfprint_b200 import HashTable
    return HashTable(path)


def test_reference_cli_runs_on_the_mirror_classes(tmp_path, golden_match):
    gm = golden_match
    from audfprint_b200.analyzer import hashes_save
    names = []
    for i in range(10):                      # precomputed fingerprints of ten reference tracks
        fn = str(tmp_path / ("trk%02d.afpt" % i))
        hashes_save(fn, gm["track%d/hashes" % i])
        names.append(fn)
    dbs = {}
    for tag, swap in (("mirror", True), ("ref", False)):
        a, b, c = (str(tmp_path / ("%s_%s.pklz" % (tag, x))) for x in "abc")
        # tiny geometry so that buckets overflow (random replacement, seeded per command)
        geo = ["--hashbits", "10", "--bucketsize", "6", "--maxtimebits", "12"]
        cmds = [["new", "--dbase", a] + geo + names[:5],
                ["add", "--dbase", a] + names[5:7],
                ["new", "--dbase", b] + geo + names[7:],
                ["remove", "--dbase", a, names[1]],
                ["newmerge", "--dbase", c] + geo + [a, b],
                ["list", "--dbase", c]]
        out = _run(str(tmp_path), swap, cmds)
        dbs[tag] = (a, b, c, out)
    for k in range(3):
        m, r = _load_db(dbs["mirror"][k]), _load_db(dbs["ref"][k])
        strip = lambda ns: [n and os.path.basename(n) for n in ns]          # noqa: E731
        assert strip(m.names) == strip(r.names)
        assert np.array_equal(m.counts, r.counts), k
        assert np.array_equal(m.table, r.table), k
        assert np.array_equal(m.hashesperid, r.hashesperid), k
        assert (m.hashbits, m.depth, m.maxtimebits) == (r.hashbits, r.depth, r.maxtimebits) == (10, 6, 12)
    # the `list` report and the bookkeeping lines are the same text (paths aside)
    norm = lambda s: [re.sub(r"(mirror|ref)_", "", ln) for ln in s.splitlines()      # noqa: E731
                      if ln.startswith(("Saved", "Read", "Removed")) or "hashes)" in ln]
    assert norm(dbs["mirror"][3]) == norm(dbs["ref"][3]) and len(norm(dbs["ref"][3])) > 10
    # and the reference itself loads what the mirror wrote
    out = _run(str(tmp_path), False, [["list", "--dbase", dbs["mirror"][2]]])
    assert "trk00.afpt" in out and "trk09.afpt" in out


def test_reference_multiprocess_add_on_the_mirror_classes(tmp_path, golden_match):
    """`new --ncores 2` (audfprint.py:199-235): the reference forks one process per file list,
    each builds a table of the swapped-in class, pickles it back through a pipe and the parent
    merges them - the mirror objects have to survive that round trip (SURVEY.md 8b, threading /
    processes) and give the table the pure reference gives.  Geometry: 37 slots hold every bucket
    of either child (CPython reseeds `random` in a forked child, so overflow draws THERE differ
    from run to run in the reference itself), while four buckets of the merged table overflow and
    take the parent's seeded np.random.permutation draws (hash_table.py:309-313)."""
    gm = golden_match
    from audfprint_b200.analyzer import hashes_save
    names = []
    for i in range(10):
        fn = str(tmp_path / ("mp%02d.afpt" % i))
        hashes_save(fn, gm["track%d/hashes" % i])
        names.append(fn)
    geo = ["--hashbits", "10", "--bucketsize", "37", "--maxtimebits", "12"]
    out = {}
    for tag, swap in (("mirror", True), ("ref", False)):
        db = str(tmp_path / (tag + "_mp.pklz"))
        text = _run(str(tmp_path), swap, [["new", "--dbase", db, "--ncores", "2"] + geo + names])
        out[tag] = (_load_db(db), text)
    m, r = out["mirror"][0], out["ref"][0]
    assert m.names == r.names and len(m.names) == 10
    assert m.names[:5] == names[0::2] and m.names[5:] == names[1::2]        # the ix % ncores deal, core by core
    assert np.array_equal(m.counts, r.counts) and np.array_equal(m.table, r.table)
    assert np.array_equal(m.hashesperid, r.hashesperid)
    assert int(np.sum(r.counts > 37)) == 4                                    # the merge did overflow
    lines = lambda s: [ln for ln in s.splitlines() if ln.startswith("hash_table ")]     # noqa: E731
    assert lines(out["mirror"][1]) == lines(out["ref"][1]) and len(lines(out["ref"][1])) == 2
