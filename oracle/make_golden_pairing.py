"""Golden vectors for tests/test_oracle_pairing.py: what the reference's analyzer produces with the
pairing window (mindt / targetdt / targetdf) and fan-out at the limits of the 6-bit hash fields, and
what its peaks2landmarks makes of explicit peak lists whose columns lie beyond 2^20, 2^21 and 2^22.
The reference is imported in a subprocess, as in make_golden_live.py.

Needs a checkout of the reference:
    AFP_REFERENCE=<checkout> python oracle/make_golden_pairing.py
Only OUTPUT ARRAYS of the reference (and the seeded peak lists it was given) are stored; no reference
source is copied.
"""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle.make_golden_live import run  # noqa: E402
from tests import cases  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "pairing.npz")

_DRIVER = r'''
import json, sys
import numpy as np
sys.path.insert(0, %(root)r); sys.path.insert(0, %(ref)r)
import audfprint_analyze as an, audio_read as ar
from audfprint_b200.synth import pcm_to_float
from tests import cases
pcm = {}
ar.audio_read = lambda fn, sr=None, channels=None: (pcm_to_float(pcm[fn]), 11025)
out = {}
tracks = cases.pairing_tracks()
for k, (mindt, targetdt, targetdf, fanout, maxpks, shifts, density, f_sd) in enumerate(cases.PAIRING_SETTINGS):
    for i, t in enumerate(tracks):
        pcm["t"] = t
        a = an.Analyzer(density)
        a.mindt, a.targetdt, a.targetdf, a.maxpairsperpeak = mindt, targetdt, targetdf, fanout
        a.maxpksperframe, a.shifts, a.f_sd = maxpks, shifts, f_sd
        out["h/%%d/%%d" %% (k, i)] = np.asarray(a.wavfile2hashes("t")).reshape(-1, 2).tolist()
        out["p/%%d/%%d" %% (k, i)] = np.asarray(a.wavfile2peaks("t")).reshape(-1, 2).tolist()
for m, (mindt, targetdt, targetdf, fanout, maxpks) in enumerate(cases.PEAK_LIST_SETTINGS):
    a = an.Analyzer()
    a.mindt, a.targetdt, a.targetdf, a.maxpairsperpeak, a.maxpksperframe = mindt, targetdt, targetdf, fanout, maxpks
    for j, start in enumerate(cases.PEAK_LIST_STARTS):
        pk = cases.peak_list(100 * m + j, start, maxpks)
        out["lists/%%d/%%d/peaks" %% (m, j)] = pk.tolist()
        lms = a.peaks2landmarks([(int(c), int(b)) for c, b in pk])
        out["lists/%%d/%%d/landmarks" %% (m, j)] = np.asarray(lms, np.int64).reshape(-1, 4).tolist()
print("JSON" + json.dumps(out))
'''


def main():
    ref = os.environ["AFP_REFERENCE"]
    g = {k: np.array(v, np.int32).reshape(-1, 4 if k.endswith("landmarks") else 2)
         for k, v in run(_DRIVER % {"root": ROOT, "ref": ref}).items()}
    np.savez_compressed(OUT, **g)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
