"""CPU: the oracle against what the reference produced with the pairing window at the limits of the
6-bit hash fields and on peak lists beyond column 2^20 (tests/golden/pairing.npz, written by
oracle/make_golden_pairing.py from a checkout of the reference).  tests/test_gpu_landmarks.py checks
the CUDA path against the oracle on the same inputs."""
import os

import numpy as np
import pytest

from audfprint_b200.synth import pcm_to_float
from oracle import afp_oracle as orc
from tests import cases
from tests.conftest import GOLDEN


@pytest.fixture(scope="module")
def golden_pairing():
    return np.load(os.path.join(GOLDEN, "pairing.npz"))


@pytest.mark.parametrize("k", range(len(cases.PAIRING_SETTINGS)))
def test_oracle_equals_reference_on_pairing_settings(golden_pairing, k):
    mindt, targetdt, targetdf, fanout, maxpks, shifts, density, f_sd = cases.PAIRING_SETTINGS[k]
    for i, t in enumerate(cases.pairing_tracks()):
        d = pcm_to_float(t)
        got = orc.fingerprint(d, density=density, fanout=fanout, shifts=shifts, f_sd=f_sd, maxpks=maxpks,
                              mindt=mindt, targetdt=targetdt, targetdf=targetdf)
        assert np.array_equal(got, golden_pairing["h/%d/%d" % (k, i)]), i
        pk = np.array(orc.find_peaks(d, density=density, f_sd=f_sd, maxpks=maxpks), np.int32).reshape(-1, 2)
        assert np.array_equal(pk, golden_pairing["p/%d/%d" % (k, i)]), i


@pytest.mark.parametrize("m", range(len(cases.PEAK_LIST_SETTINGS)))
def test_oracle_peaks_to_landmarks_equals_reference_past_2_20_columns(golden_pairing, m):
    mindt, targetdt, targetdf, fanout, maxpks = cases.PEAK_LIST_SETTINGS[m]
    for j, start in enumerate(cases.PEAK_LIST_STARTS):
        pk = golden_pairing["lists/%d/%d/peaks" % (m, j)]
        assert np.array_equal(pk, cases.peak_list(100 * m + j, start, maxpks)), j
        # full columns, an empty stretch longer than the window, a lone final peak
        assert np.bincount(pk[:, 0] - start).max() == maxpks
        assert np.diff(pk[:, 0]).max() > targetdt and pk[-1, 0] > pk[-2, 0]
        got = orc.peaks_to_landmarks([(int(c), int(b)) for c, b in pk], fanout, mindt, targetdt, targetdf)
        want = golden_pairing["lists/%d/%d/landmarks" % (m, j)]
        assert np.array_equal(np.array(got, np.int32).reshape(-1, 4), want), j
