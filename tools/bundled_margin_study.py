"""How far are the decisions made on the bundled real-music fixtures (tests/golden/bundled_pcm.npz)
from flipping?  The CUDA spectrogram differs from NumPy's by last-ulp rounding (|d| ~ 1e-15..1e-13
of the largest bin; tests assert <= 1e-11).  This CPU study adds complex Gaussian noise of EPS times
the largest STFT bin to the oracle's STFT and counts fingerprints that change: the committed PCM
(query, four tracks, four excerpts) x densities {100, 20} x shifts {1, 4} x 3 draws.

    python tools/bundled_margin_study.py 1e-12 1e-10      # -> profiles/r02_bundled_margin_study.json
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import afp_oracle as orc      # noqa: E402  (test infrastructure, CPU only)


def main():
    g = np.load(os.path.join(ROOT, "tests", "golden", "bundled_pcm.npz"))
    sigs = {"query": g["query/pcm"]}
    for k in (0, 4, 8, 12):
        sigs["track%d" % k] = g["track%d/pcm" % k]
        sigs["excerpt%d" % k] = g["track%d/pcm" % k][3 * 11025:8 * 11025]
    exact = orc.stft_complex
    out = []
    for eps in [float(x) for x in sys.argv[1:]] or [1e-12]:
        rng = np.random.default_rng(1)

        def noisy(d, *a, **k):
            X = exact(d, *a, **k)
            return X + eps * np.max(np.abs(X)) * (rng.standard_normal(X.shape) + 1j * rng.standard_normal(X.shape))
        flips = total = 0
        for name, pcm in sigs.items():
            d = pcm.astype(np.float32) / 32768.0
            for dens in (100.0, 20.0):
                for sh in (1, 4):
                    orc.stft_complex = exact
                    base = orc.fingerprint(d, density=dens, shifts=sh)
                    orc.stft_complex = noisy
                    for _ in range(3):
                        total += 1
                        flips += not np.array_equal(orc.fingerprint(d, density=dens, shifts=sh), base)
        orc.stft_complex = exact
        out.append({"eps_of_largest_bin": eps, "fingerprints": total, "changed": int(flips)})
        print(out[-1])
    with open(os.path.join(ROOT, "profiles", "r02_bundled_margin_study.json"), "w") as f:
        json.dump({"what": __doc__.strip().split("\n\n")[0], "results": out}, f, indent=1)


if __name__ == "__main__":
    main()
