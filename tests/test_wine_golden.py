"""Stage (c), SURVEY 8 row a15: the band integration restated in oracle/oracle.py
(readfilter / resample / bandintegrate) and the host precompute the CUDA path uses
(bart_b200.api.filters_from_files) against what the reference's own code/wine.py:16-66,127-199
returns (tests/golden/wine.npz, written by tests/golden/make_golden_wine.py from the imported
reference module; filters and Kurucz model as shipped in the reference's inputs/)."""
import os

import numpy as np
import pytest

from oracle import oracle as orc

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "wine.npz"))
SETS = {"demo": 10, "w12": 4}


def write_filter(path, fwn, ftr):
    """A filter file in the reference's format (wavelength in microns, response), holding the same
    (wavenumber, response) pairs the golden recorded -- the reference's inputs/ do not travel."""
    wl = 1.0 / (fwn * 1e-4)
    with open(path, "w") as f:
        f.write("# wavelength (um)  response\n\n")
        for a, b in zip(wl[::-1], ftr[::-1]):
            f.write("%.17g %.17g\n" % (a, b))


@pytest.mark.parametrize("name", list(SETS))
def test_oracle_resample_bandintegrate(name, tmp_path):
    specwn, spectrum = G[name + "_specwn"], G[name + "_spectrum"]
    for i in range(SETS[name]):
        key = "%s_%d_" % (name, i)
        path = str(tmp_path / ("f%d.dat" % i))
        write_filter(path, G[key + "fwn"], G[key + "ftr"])
        fwn, ftr = orc.readfilter(path)
        # 17 significant digits through 1/(wl 1e-4): the wavenumbers come back to the last bit or two
        assert np.allclose(fwn, G[key + "fwn"], rtol=4e-16, atol=0)
        assert np.array_equal(ftr, G[key + "ftr"])
        nif, istar, idx = orc.resample(specwn, G[key + "fwn"], G[key + "ftr"], G["starwn"], G["starfl"])
        assert np.array_equal(idx, G[key + "idx"])
        assert np.allclose(nif, G[key + "nifilter"], rtol=1e-13, atol=0)
        assert np.allclose(istar, G[key + "istarfl"], rtol=1e-13, atol=0)
        be = orc.bandintegrate(spectrum[idx] / istar * 0.117 ** 2, specwn, nif, idx)
        bt = orc.bandintegrate(spectrum[idx], specwn, nif, idx)
        assert abs(be / G[key + "band_eclipse"] - 1) < 1e-13
        assert abs(bt / G[key + "band_transit"] - 1) < 1e-13


@pytest.mark.parametrize("name", list(SETS))
def test_api_filters_from_files(name, tmp_path):
    """The precompute that feeds K4 (start, count, weights, star) = wine.resample's outputs."""
    from bart_b200 import api
    specwn = G[name + "_specwn"]
    files = []
    for i in range(SETS[name]):
        key = "%s_%d_" % (name, i)
        files.append(str(tmp_path / ("f%d.dat" % i)))
        write_filter(files[-1], G[key + "fwn"], G[key + "ftr"])
    start, count, weight, star = api.filters_from_files(specwn, files, G["starwn"], G["starfl"])
    off = 0
    for i in range(SETS[name]):
        key = "%s_%d_" % (name, i)
        idx = G[key + "idx"]
        assert start[i] == idx[0] and count[i] == len(idx)
        assert np.allclose(weight[off:off + count[i]], G[key + "nifilter"], rtol=1e-12, atol=0)
        assert np.allclose(star[off:off + count[i]], G[key + "istarfl"], rtol=1e-12, atol=0)
        # K4's formula (kernels.cu band_integrate_kernel) in numpy on the same arrays
        y = G[name + "_spectrum"][idx] / star[off:off + count[i]] * 0.117 ** 2 * weight[off:off + count[i]]
        band = 0.5 * np.sum(np.diff(specwn[idx]) * (y[1:] + y[:-1]))
        assert abs(band / G[key + "band_eclipse"] - 1) < 1e-12
        off += count[i]


def test_read_kurucz_vs_reference():
    """api.read_kurucz against wine.readkurucz (golden wine.npz) on a shrunk copy of the Kurucz grid
    the reference ships (tests/golden/make_golden_kurucz.py: the selected model restated digit for
    digit from the golden, between placeholder neighbours)."""
    from bart_b200 import api
    kfile = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kurucz_t6000g45.pck")
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "wine.npz"))
    starfl, starwn, tmodel, gmodel = api.read_kurucz(kfile, 6000.0, 4.5)
    assert np.array_equal(starwn, g["starwn"]) and np.array_equal(starfl, g["starfl"])
    assert (tmodel, gmodel) == tuple(g["star_model"])
