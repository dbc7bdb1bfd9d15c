"""GPU: retrievals with polar (Rayleigh, polarizability) scattering -- `scattering = polar` in the
[MCMC] section, nray = 2 -- against the retrieval oracle.  The scattering model takes one parameter
slot whose value is unused, so the abundance factors follow it; `small4` with all four molecules
fitted makes a shift between molecules visible."""
import os
import subprocess
import sys

import numpy as np
import pytest

import cases
from util import relerr

pytestmark = pytest.mark.gpu
MOLFIT = ("H2O", "CO2", "CO", "CH4")
NPT, ICLOUD, IPOLAR = 5, 5, 6          # [PT x5 | cloud top | polar slot | 4 abundance factors]
NOMINAL = [-0.5, -0.2, 1.0, 0.0, 1.1, -1.0, 0.0, 0.0, 0.5, -0.5, 0.2]
PMIN = [-5.0, -3.0, -2.0, 0.0, 0.55, -4.0, -9.0, -9.0, -9.0, -9.0, -9.0]
PMAX = [2.0, 2.0, 3.0, 1.0, 1.4, 1.5, 3.0, 3.0, 3.0, 3.0, 3.0]
RPRS = 0.117


@pytest.fixture(scope="module")
def api(built):
    from bart_b200 import api as a
    a.lib()
    return a


def black_body_star(wn):
    starwn = np.linspace(wn[0] - 10, wn[-1] + 10, 3000)
    hc_k = 6.6260755e-27 * 2.99792458e10 / 1.380658e-16
    return starwn, 2 * 6.6260755e-27 * 2.99792458e10 ** 2 * starwn ** 3 / np.expm1(hc_k * starwn / 6300.0)


@pytest.fixture(scope="module")
def polar(workdir):
    from bart_b200 import synth
    case = synth.make_case(os.path.join(workdir, "polar_small4"), shape="small4", solution="eclipse",
                           seed=2033, nlayer=60)
    starwn, starfl = black_body_star(case["wn"])
    return case, starwn, starfl


def converter(case):
    from oracle import retrieval_oracle as ro
    return ro.Converter(case["press_bar"], case["species"], case["abund"], MOLFIT, "line",
                        pt_args=cases.W12_PTARGS, ncloud=1, nray=2)


def setup(api, polar):
    case, starwn, starfl = polar
    tr = api.Transit(case["cfg"])
    wn = tr.get_waveno_arr()
    tr.set_filters(*api.filters_from_files(wn, case["filters"], starwn, starfl), RPRS)
    npars = tr.converter_init(case["press_bar"], case["species"], case["abund"], MOLFIT, "line",
                              pt_args=cases.W12_PTARGS, nrad=0, ncloud=1, nray=2)
    assert npars == len(NOMINAL)
    return tr


def draws(seed=9):
    """Accepted proposals, temperature-bound rejections and abundance rejections."""
    rng = np.random.default_rng(seed)
    p = rng.uniform(PMIN, PMAX, (32, len(NOMINAL)))
    p[:, NPT + 2:] = rng.uniform(-2.0, 1.0, (32, 4))
    p[:24, :NPT] = np.array(NOMINAL[:NPT]) + rng.normal(0, 0.02, (24, NPT))
    p[[3, 9, 15], -2] = 4.2                                  # CO2: metals past 1
    p[[4, 10], -4] = 4.2                                     # H2O
    return p


def test_polar_profiles_vs_oracle(api, polar):
    case = polar[0]
    tr = setup(api, polar)
    params = draws()
    prof, status, knobs = tr.profiles_from_params(params)
    oprof, ostatus, oknobs = converter(case).profiles(params)
    assert np.array_equal(status, ostatus)
    ok = status == 0
    assert ok.sum() >= 8 and (status == api.REJ_TBOUNDS).any() and (status == api.REJ_ABUND).any()
    assert relerr(prof[ok], oprof[ok]) < 1e-13
    assert np.array_equal(knobs[1], params[:, ICLOUD])
    assert np.all(knobs[2] == 0.0) and np.all(oknobs["scat_flag"] == 2)
    # the polar slot's value changes nothing, bit for bit
    for v in (-9.0, 3.0, 1e300):
        q = params.copy()
        q[:, IPOLAR] = v
        prof2, status2, knobs2 = tr.profiles_from_params(q)
        assert np.array_equal(prof2, prof) and np.array_equal(status2, status)
        assert np.array_equal(knobs2, knobs)
    tr.free_memory()


def test_polar_bandflux_vs_oracle(api, polar):
    from oracle import retrieval_oracle as ro
    case, starwn, starfl = polar
    tr = setup(api, polar)
    params = draws(10)
    bf, status = tr.bandflux_from_params(params)
    band = ro.BandOracle(case["cfg"], converter(case), case["filters"], starwn, starfl, RPRS)
    ref = band(params)
    _, ostatus, _ = band.conv.profiles(params)
    assert np.array_equal(status, ostatus)
    ok = status == 0
    assert ok.sum() >= 8 and np.all(bf[~ok] == -1.0) and np.all(ref[~ok] == -1.0)
    assert relerr(bf[ok], ref[ok]) < 1e-8
    # the converter hands the forward model scat_flag 2 for every model: the same band fluxes and
    # scattering extinction as the host path with that knob set explicitly
    n = int(ok.sum())
    bf1, _ = tr.bandflux_from_params(params[ok])
    scat1 = tr.debug_get("scat", n - 1)
    prof, _, knobs = tr.profiles_from_params(params[ok])
    tr.set_batch_knobs(n, cloudtop=knobs[1], scat_flag=np.full(n, 2, np.int32), scat_logext=np.zeros(n))
    bf2, _ = tr.bandflux_batch(prof)
    tr.set_batch_knobs(0)
    assert np.array_equal(bf2, bf1) and np.array_equal(bf1, bf[ok])
    assert np.array_equal(tr.debug_get("scat", n - 1), scat1) and np.all(scat1 > 0)
    tr.free_memory()


_demc_ref = {}


@pytest.mark.parametrize("graph", ["1", "0"])
def test_polar_demc_on_device_vs_oracle(graph, api, polar, monkeypatch):
    """A short DE-MC run on the device against retrieval_oracle.demc on the same seeded streams."""
    from bart_b200 import driver
    from oracle import retrieval_oracle as ro
    monkeypatch.setenv("BART_MCMC_GRAPH", graph)
    case, starwn, starfl = polar
    band = ro.BandOracle(case["cfg"], converter(case), case["filters"], starwn, starfl, RPRS)
    truth = np.array([-0.6, -0.15, 1.0, 0.0, 1.08, -0.8, 0.0, 0.3, 0.2, -0.3, 0.0])
    data = band(truth)[0]
    uncert = 0.02 * np.abs(data)
    stepsize = np.array([0.05, 0.05, 0.0, 0.0, 0.01, 0.2, 0.0, 0.3, 0.3, 0.3, 0.3])
    nchains, numit, seed = 6, 360, 4242
    tr = setup(api, polar)
    np.random.seed(seed)
    out = driver.run_demc(tr, data, uncert, NOMINAL, PMIN, PMAX, stepsize, numit, nchains)
    if "ref" not in _demc_ref:
        np.random.seed(seed)
        _demc_ref["ref"] = ro.demc(band, data, uncert, NOMINAL, PMIN, PMAX, stepsize, numit, nchains)
    ref = _demc_ref["ref"]
    assert out["allparams"].shape == (nchains, int((stepsize > 0).sum()), numit // nchains)
    assert np.array_equal(out["allparams"], ref["allparams"])
    assert np.array_equal(out["bestp"], ref["bestp"])
    assert np.array_equal(out["numaccept"], ref["numaccept"])
    assert 0 < ref["numaccept"].sum() < numit
    tr.free_memory()


def test_bartworker_with_polar_scattering(api, polar, workdir):
    """driver.BartWorker from an [MCMC] section with `scattering = polar`, against the band oracle."""
    from bart_b200 import driver
    from oracle import retrieval_oracle as ro
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_golden_bartfunc as gen
    case, starwn, starfl = polar
    tepfile = os.path.join(workdir, "polar_planet.tep")
    with open(tepfile, "w") as f:
        f.write(gen.TEP)
    cfg = os.path.join(workdir, "polar_MCMC.cfg")
    with open(cfg, "w") as f:
        f.write("[MCMC]\n")
        f.write("molfit = %s\n" % " ".join(MOLFIT))
        f.write("atmfile = %s\nPTtype = line\ntint = 100.0\ntint_type = const\n" % case["atm"])
        f.write("tconfig = %s\n" % case["cfg"])
        f.write("filters = %s\n" % "\n    ".join(case["filters"]))
        f.write("tep_name = %s\nsolution = eclipse\nscattering = polar\n" % tepfile)
    w = driver.BartWorker(cfg, star=(starwn, starfl))
    assert w.npars == NPT + 1 + len(MOLFIT)
    sysp = driver.system_from_tep(tepfile, tint=100.0)
    species, press, _, abund = driver.read_atm(case["atm"])
    conv = ro.Converter(press, species, abund, MOLFIT, "line", pt_args=sysp["pt_args"], nray=2)
    band = ro.BandOracle(case["cfg"], conv, case["filters"], starwn, starfl, sysp["rprs"])
    params = np.delete(draws(11), ICLOUD, axis=1)             # no cloud slot in this configuration
    bf = w(params)
    ref = band(params)
    rej = ref[:, 0] == -1
    assert (~rej).sum() >= 8 and rej.any()
    assert np.all(bf[rej] == -1.0)
    assert relerr(bf[~rej], ref[~rej]) < 1e-8
    w.close()


def test_first_pt_line_conversion_of_a_process(api, polar, workdir):
    """The converter's first PT_line call in a fresh process reads the E2 table the call uploads."""
    case = polar[0]
    params = draws(12)
    inp, op = os.path.join(workdir, "polar_e2_in.npz"), os.path.join(workdir, "polar_e2_out.npz")
    np.savez(inp, params=params, press=case["press_bar"], abund=case["abund"])
    code = "\n".join([
        "import sys, numpy as np",
        "sys.path[:0] = [%r, %r]" % (cases.ROOT, os.path.join(cases.ROOT, "tests")),
        "import cases",
        "from bart_b200 import api",
        "d = np.load(%r)" % inp,
        "tr = api.Transit(%r)" % case["cfg"],
        "tr.converter_init(d['press'], %r, d['abund'], %r, 'line', pt_args=cases.W12_PTARGS, "
        "nrad=0, ncloud=1, nray=2)" % (case["species"], MOLFIT),
        "prof, status, _ = tr.profiles_from_params(d['params'])",
        "np.savez(%r, prof=prof, status=status)" % op])
    subprocess.check_call([sys.executable, "-c", code])
    got = np.load(op)
    prof, status = got["prof"], got["status"]
    oprof, ostatus, _ = converter(case).profiles(params)
    assert np.array_equal(status, ostatus)
    ok = status == 0
    assert ok.sum() >= 8 and relerr(prof[ok], oprof[ok]) < 1e-12
