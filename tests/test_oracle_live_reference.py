"""CPU: the oracle against what the reference produced on seeds and parameter settings that
the other golden files do not cover (tests/golden/live_reference.npz, written by
oracle/make_golden_live.py from a checkout of the reference)."""
import os

import numpy as np
import pytest

from audfprint_b200.synth import synth_track, synth_query, pcm_to_float
from oracle import afp_oracle as orc
from tests.conftest import GOLDEN

FRESH_SEEDS = [5101, 5102, 5103, 5104]
ANALYZER_PARAMS = [(20.0, 3, 2, 30.0, 5), (20.0, 3, 3, 30.0, 5), (20.0, 3, 8, 30.0, 5), (35.0, 5, 1, 20.0, 3),
                   (50.0, 6, 4, 30.0, 8), (10.0, 1, 1, 45.0, 1), (70.0, 8, 1, 30.0, 16)]
MATCHER_PARAMS = [(0, 5, 100, 100), (3, 0, 5, 100), (1, 5, 1, 100), (2, 1, 100, 0), (2, 5, 0, 100), (1, 2, 3, 1)]
SPREAD_CASES = [(256, 4.0), (256, 30.0), (64, 2.5), (17, 1.0), (300, 12.0), (1, 4.0)]


@pytest.fixture(scope="module")
def golden_live():
    return np.load(os.path.join(GOLDEN, "live_reference.npz"))


def outputs(g, group):
    """The stored outputs of one reference run, under the names that run gave them."""
    return {k[len(group) + 1:]: g[k] for k in g.files if k.startswith(group + "/")}


def test_oracle_equals_live_reference_on_fresh_seeds(golden_live):
    seeds = FRESH_SEEDS
    ref = outputs(golden_live, "fresh")
    tracks = []
    for seed in seeds:
        d = pcm_to_float(synth_track(seed, 14.0 + seed % 5))
        for shifts in (1, 4):
            got = orc.fingerprint(d, shifts=shifts)
            assert np.array_equal(got, np.array(ref["h_%d_%d" % (seed, shifts)], np.int32).reshape(-1, 2)), (seed, shifts)
        tracks.append(orc.fingerprint(d, shifts=1))
    import random
    rng = random.Random(4)
    t = orc.Table(hashbits=14, depth=6, maxtimebits=12)
    for i, h in enumerate(tracks):
        t.store("s%d" % i, h, rng)
    assert np.array_equal(t.table, np.array(ref["table"], np.uint32)) and np.array_equal(t.counts, ref["counts"])
    hpi = np.array(ref["hpi"])
    for j, seed in enumerate(seeds):
        q, _ = synth_query(synth_track(seed, 14.0 + seed % 5), 77 + j, seconds=6.0, noise_sigma=0.01)
        qh = orc.fingerprint(pcm_to_float(q), shifts=4)
        assert np.array_equal(qh, np.array(ref["q_%d" % seed], np.int32).reshape(-1, 2))
        hits = orc.get_hits(t.table, t.counts, 14, 6, 12, qh)
        assert np.array_equal(hits, np.array(ref["hits_%d" % seed], np.int32).reshape(-1, 4))
        rows = orc.match_hashes(t.table, t.counts, 14, 6, 12, hpi, qh, window=2, threshcount=3, search_depth=4)
        want = np.array(ref["rows_%d" % seed], np.int32).reshape(-1, 7)
        assert rows.shape == want.shape and np.array_equal(rows[:1], want[:1]), seed   # best match identical
        assert sorted(map(tuple, rows[:, :4])) == sorted(map(tuple, want[:, :4]))        # same alignments


def test_oracle_equals_live_reference_on_non_default_parameters(golden_live):
    """The parameter settings the GPU tests check against the ORACLE only
    (test_non_default_analyzer_parameters_vs_oracle, test_matcher_edge_parameters_vs_oracle) -
    density / fanout / shifts / f_sd / maxpksperframe and window / threshcount / search_depth /
    max_alignments_per_id - checked here oracle vs the reference's outputs, which closes the chain."""
    ref = outputs(golden_live, "params")
    for k, (density, fanout, shifts, f_sd, maxpks) in enumerate(ANALYZER_PARAMS):
        for i in range(2):
            d = pcm_to_float(synth_track(6000 + 10 * k + i, 9.0 + i))
            got = orc.fingerprint(d, density=density, fanout=fanout, shifts=shifts, f_sd=f_sd, maxpks=maxpks)
            assert np.array_equal(got, np.array(ref["h_%d_%d" % (k, i)], np.int32).reshape(-1, 2)), (k, i)
            if shifts == 1:
                pk = orc.find_peaks(d, density=density, f_sd=f_sd, maxpks=maxpks)
                assert np.array_equal(np.array(pk, np.int32).reshape(-1, 2),
                                      np.array(ref["p_%d_%d" % (k, i)], np.int32).reshape(-1, 2)), (k, i)
    table, counts, hpi = np.array(ref["table"], np.uint32), np.array(ref["counts"], np.int32), np.array(ref["hpi"])
    nexact = 0
    for k, (window, thresh, sdepth, maxal) in enumerate(MATCHER_PARAMS):
        for j in range(4):
            qh = np.array(ref["q_%d" % j], np.int32).reshape(-1, 2)
            want = np.array(ref["rows_%d_%d" % (k, j)], np.int32).reshape(-1, 7)
            rows = orc.match_hashes(table, counts, 12, 8, 14, hpi, qh, window=window, threshcount=thresh,
                                    search_depth=sdepth, max_alignments_per_id=maxal)
            assert rows.shape == want.shape and np.array_equal(rows[:, 1], want[:, 1]), (k, j)
            # rank order among equal weights / equal counts is implementation-defined in the reference
            assert sorted(map(tuple, rows[:, :4])) == sorted(map(tuple, want[:, :4])), (k, j)
            nexact += int(np.array_equal(rows, want))
    assert nexact >= 12


def test_spread_local_maxes_equals_reference_spreadpeaksinvector(golden_live):
    """The stand-alone method north_star names (audfprint_analyze.py:153-160): the oracle function
    the GPU test compares afp_spread_peaks with, against the reference's own method."""
    for k, (n, width) in enumerate(SPREAD_CASES):
        v, want = golden_live["spread/%d/v" % k], golden_live["spread/%d/want" % k]
        assert len(v) == n
        got = orc.spread_local_maxes(v, orc.gaussian_table(n, width))
        assert np.array_equal(got, want), (n, width)
