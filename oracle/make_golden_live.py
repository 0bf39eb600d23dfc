"""Golden vectors for tests/test_oracle_live_reference.py: what the reference's analyzer,
hash table and matcher produce on seeds and parameter settings that the other golden files
do not cover.  The reference is imported in a subprocess so that its module names
(hash_table, ...) never enter this process.

Needs a checkout of the reference:
    AFP_REFERENCE=<checkout> python oracle/make_golden_live.py
Only OUTPUT ARRAYS of the reference are stored; no reference source is copied.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests.test_oracle_live_reference import (ANALYZER_PARAMS, FRESH_SEEDS, MATCHER_PARAMS,  # noqa: E402
                                              SPREAD_CASES)

OUT = os.path.join(ROOT, "tests", "golden", "live_reference.npz")
DTYPES = {"table": np.uint32, "hpi": np.int64}

_DRIVER = r'''
import json, random, sys
import numpy as np
sys.path.insert(0, %(root)r); sys.path.insert(0, %(ref)r)
import audfprint_analyze as an, audfprint_match as ma, audio_read as ar, hash_table as htm
from audfprint_b200.synth import synth_track, synth_query, pcm_to_float
pcm = {}
ar.audio_read = lambda fn, sr=None, channels=None: (pcm_to_float(pcm[fn]), 11025)
out = {}
tracks = []
for seed in %(seeds)r:
    pcm["t"] = synth_track(seed, 14.0 + seed %% 5)
    for shifts in (1, 4):
        a = an.Analyzer(); a.shifts = shifts
        out["h_%%d_%%d" %% (seed, shifts)] = np.asarray(a.wavfile2hashes("t")).tolist()
    tracks.append(np.asarray(out["h_%%d_1" %% seed], np.int32))
random.seed(4)
ht = htm.HashTable(hashbits=14, depth=6, maxtime=1 << 12)
for i, h in enumerate(tracks):
    ht.store("s%%d" %% i, h)
m = ma.Matcher(); m.window = 2; m.threshcount = 3; m.search_depth = 4
for j, seed in enumerate(%(seeds)r):
    q, _ = synth_query(synth_track(seed, 14.0 + seed %% 5), 77 + j, seconds=6.0, noise_sigma=0.01)
    pcm["q"] = q
    a = an.Analyzer(); a.shifts = 4
    qh = np.asarray(a.wavfile2hashes("q"), np.int32)
    out["q_%%d" %% seed] = qh.tolist()
    out["hits_%%d" %% seed] = ht.get_hits(qh).tolist()
    out["rows_%%d" %% seed] = m.match_hashes(ht, qh).tolist()
out["table"] = ht.table.tolist(); out["counts"] = ht.counts.tolist(); out["hpi"] = np.asarray(ht.hashesperid).tolist()
print("JSON" + json.dumps(out))
'''

_PARAM_DRIVER = r'''
import json, random, sys
import numpy as np
sys.path.insert(0, %(root)r); sys.path.insert(0, %(ref)r)
import audfprint_analyze as an, audfprint_match as ma, audio_read as ar, hash_table as htm
from audfprint_b200.synth import synth_track, synth_query, pcm_to_float
pcm = {}
ar.audio_read = lambda fn, sr=None, channels=None: (pcm_to_float(pcm[fn]), 11025)
out = {}
for k, (density, fanout, shifts, f_sd, maxpks) in enumerate(%(aparams)r):
    for i in range(2):
        pcm["t"] = synth_track(6000 + 10 * k + i, 9.0 + i)
        a = an.Analyzer(density)
        a.maxpairsperpeak, a.shifts, a.f_sd, a.maxpksperframe = fanout, shifts, f_sd, maxpks
        out["h_%%d_%%d" %% (k, i)] = np.asarray(a.wavfile2hashes("t")).reshape(-1, 2).tolist()
        if shifts == 1:
            out["p_%%d_%%d" %% (k, i)] = np.asarray(a.wavfile2peaks("t")).reshape(-1, 2).tolist()
# matcher parameters on a small overflowing table
random.seed(9)
ht = htm.HashTable(hashbits=12, depth=8, maxtime=1 << 14)
trk = [synth_track(6500 + i, 12.0) for i in range(12)]
for i, t in enumerate(trk):
    pcm["t"] = t
    ht.store("s%%d" %% i, an.Analyzer().wavfile2hashes("t"))
out["table"] = ht.table.tolist(); out["counts"] = ht.counts.tolist(); out["hpi"] = np.asarray(ht.hashesperid).tolist()
qs = []
for j in range(4):
    q, _ = synth_query(trk[3 * j], 900 + j, seconds=7.0, noise_sigma=0.01)
    pcm["q"] = q
    a = an.Analyzer(); a.shifts = 4
    qs.append(np.asarray(a.wavfile2hashes("q"), np.int32).reshape(-1, 2))
    out["q_%%d" %% j] = qs[-1].tolist()
for k, (window, thresh, sdepth, maxal) in enumerate(%(mparams)r):
    m = ma.Matcher()
    m.window, m.threshcount, m.search_depth, m.max_alignments_per_id = window, thresh, sdepth, maxal
    for j, qh in enumerate(qs):
        out["rows_%%d_%%d" %% (k, j)] = np.asarray(m.match_hashes(ht, qh)).reshape(-1, 7).tolist()
print("JSON" + json.dumps(out))
'''

_SPREAD_DRIVER = r'''
import json, sys
import numpy as np
sys.path.insert(0, %(ref)r)
import audfprint_analyze as an
rng = np.random.default_rng(12)
out = []
for n, width in %(cases)r:
    v = rng.standard_normal(n) * 3
    v[rng.integers(0, n, max(1, n // 9))] = 2.0          # plateaus / equal neighbours
    out.append([v.tolist(), an.Analyzer().spreadpeaksinvector(v, width).tolist()])
print("JSON" + json.dumps(out))
'''


def run(code):
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("JSON")][0][4:])


def main():
    ref = os.environ["AFP_REFERENCE"]
    g = {}
    fresh = run(_DRIVER % {"root": ROOT, "ref": ref, "seeds": FRESH_SEEDS})
    for k, v in fresh.items():
        g["fresh/" + k] = np.array(v, DTYPES.get(k, np.int32))
    par = run(_PARAM_DRIVER % {"root": ROOT, "ref": ref, "aparams": ANALYZER_PARAMS, "mparams": MATCHER_PARAMS})
    for k, v in par.items():
        g["params/" + k] = np.array(v, DTYPES.get(k, np.int32))
    for k, (v, want) in enumerate(run(_SPREAD_DRIVER % {"ref": ref, "cases": SPREAD_CASES})):
        g["spread/%d/v" % k] = np.array(v, np.float64)
        g["spread/%d/want" % k] = np.array(want, np.float64)
    np.savez_compressed(OUT, **g)
    print("wrote", OUT, os.path.getsize(OUT), "bytes")


if __name__ == "__main__":
    main()
