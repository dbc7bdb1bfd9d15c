#!/usr/bin/env python
"""tests/golden/kurucz_t6000g45.pck: a shrunk Kurucz grid in the layout of the reference's
inputs/kurucz/fp00k2odfnew.pck (11.8 MB, not redistributed here), for the api.read_kurucz test.

The T = 6000 K, log g = 4.5 block is that file's model restated digit for digit: its wavelengths
(nm) and line-blanketed fluxes are recovered from what wine.readkurucz returned for it
(wine.npz: starwn, starfl), and each recovered decimal is checked to map back to the stored
float64 through read_kurucz's own unit conversions bit for bit.  Around it sit placeholder models
(zero fluxes) at the neighbouring temperatures and gravities, so the nearest-model selection has
something to choose from; the continuum lines of every block are zeros (read_kurucz skips them).

    python tests/golden/make_golden_kurucz.py
"""
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "kurucz_t6000g45.pck")
C_LIGHT = 299792458.0
MODELS = [(5750.0, 4.5), (6000.0, 4.0), (6000.0, 4.5), (6000.0, 5.0), (6250.0, 4.5)]
TARGET = (6000.0, 4.5)
PER_LINE = 8


def to_starfl(v):
    """read_kurucz's flux conversion, operation for operation."""
    return v * (4.0 * 1e-3) * 1e3 * np.pi * (1e2 * C_LIGHT)


def shortest(x, fwd, target):
    """The shortest decimal (at most 10 characters) that fwd maps to exactly `target`."""
    for nd in range(1, 9):
        s = "%.*E" % (nd - 1, x)
        if len(s) <= 10 and fwd(float(s)) == target:
            return float(s)
    raise SystemExit("no 10-character decimal reproduces %r" % target)


def block(values, fmt):
    rows = []
    for i in range(0, len(values), PER_LINE):
        rows.append("".join(fmt % v for v in values[i:i + PER_LINE]))
    return rows


def main():
    g = np.load(os.path.join(HERE, "wine.npz"))
    assert tuple(g["star_model"]) == TARGET
    wn, fl = g["starwn"][::-1], g["starfl"][::-1]          # file order: ascending wavelength
    wave = [shortest(1e7 / w, lambda v: (C_LIGHT / (v * 1e-9)) / C_LIGHT * 1e-2, w) for w in wn]
    flux = [shortest(f / to_starfl(1.0), to_starfl, f) for f in fl]
    wave_rows = block(wave, "%10.2f")
    flux_rows = block(flux, "%10.4E")
    zero_rows = block([0.0] * len(flux), "%10.4E")
    # the fixed formats must not lose a digit of the recovered decimals
    assert [float(s) for r in wave_rows for s in (r[j:j + 10] for j in range(0, len(r), 10))] == wave
    assert [float(s) for r in flux_rows for s in (r[j:j + 10] for j in range(0, len(r), 10))] == flux
    lines = ["      PROGRAM READ_FLUXES", "C     layout: wavelengths (nm), then per model TEFF/GRAVITY,",
             "C     Eddington fluxes and continuum fluxes, 8 fields of 10 characters per line", "      END"]
    lines += wave_rows
    for teff, logg in MODELS:
        lines.append("TEFF %6.0f.  GRAVITY%8.5f LTE" % (teff, logg))
        lines += flux_rows if (teff, logg) == TARGET else zero_rows
        lines += zero_rows
    with open(OUT, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("wrote %s (%d bytes, %d wavelengths, %d models)" % (OUT, os.path.getsize(OUT), len(wave), len(MODELS)))


if __name__ == "__main__":
    main()
