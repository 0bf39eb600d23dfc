import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden_fp():
    return np.load(os.path.join(GOLDEN, "fingerprint.npz"))


def load_golden(*names):
    """The arrays of tests/golden/<name>.npz for every name, in one mapping (a set of vectors is
    split over several files to keep each of them under 1 MB)."""
    out = {}
    for name in names:
        with np.load(os.path.join(GOLDEN, name + ".npz")) as g:
            out.update((k, np.asarray(g[k], order="C")) for k in g.files)
    return out


@pytest.fixture(scope="session")
def golden_match():
    return load_golden("match", "match_hits")


@pytest.fixture(scope="session")
def golden_options():
    """Reference Matcher output with exact_count / find_time_range / hashesfor
    (oracle/make_golden_options.py)."""
    return np.load(os.path.join(GOLDEN, "match_options.npz"))


def option_ties(hits, hpi, rows, thresh, sdepth):
    """(candidate order ambiguous, row order ambiguous) for one reference result."""
    ids, raw = np.unique(hits[:, 0], return_counts=True)
    wtd = raw / np.asarray(hpi)[ids].astype(float)
    dep = min(int(np.count_nonzero(raw > thresh)), sdepth)
    srt = np.sort(wtd)[::-1][:dep + 1]
    return bool(dep and np.any(srt[:-1] == srt[1:])), bool(len(np.unique(rows[:, 1])) != len(rows))


def expand_table(gm, db):
    """Rebuild dense (table, counts) arrays from the sparse golden storage."""
    hashbits, depth, mtb = (int(x) for x in gm[db + "/params"])
    table = np.zeros((1 << hashbits, depth), np.uint32)
    counts = np.zeros(1 << hashbits, np.int32)
    b = gm[db + "/buckets"]
    table[b] = gm[db + "/rows"]
    counts[b] = gm[db + "/counts"]
    return table, counts, hashbits, depth, mtb, gm[db + "/hashesperid"]
