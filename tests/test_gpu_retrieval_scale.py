"""GPU: the device retrieval loop at the sizes a BART retrieval runs at, against the retrieval
oracle.  The golden-driven cases (tests/cases.py RETRIEVAL) have 4 or 10 data points, 5 or 6 chains,
no priors, the default fgamma / fepsilon and at most 37 history rows; here:

* 40 data points: more than the 32 lanes that add a chain's residuals, and not a multiple of 32;
* a Gaussian prior on kappa and a Jeffreys prior on beta (the only path where the chi-squared a
  chain walks on and the one the best fit is chosen on differ);
* fgamma 0.8 and fepsilon 0.02 (with fepsilon 0 a wrong index into `support` is multiplied by 0);
* 37 DE-MC chains: five 8-chain proposal CTAs, the last one partial, and more chains than a warp
  for the Metropolis and best-fit loops;
* a 2500-iteration snooker run whose history outgrows its reservation twice, between the grtest
  segments, with generated rows to carry over;
* band integration over filters of 2 to 2501 samples (one to five 512-trapezoid passes)."""
import os

import numpy as np
import pytest

import cases
from util import relerr

pytestmark = pytest.mark.gpu
SPEC = cases.RETRIEVAL["retr_tiny_eclipse"]      # PT_line + CH4: kappa g1 g2 alpha beta log(CH4)
MOLFIT = SPEC["molfit"]
PARAMS, PMIN, PMAX = (np.array(SPEC[k], dtype=float) for k in ("params", "pmin", "pmax"))
STEPSIZE = np.array(SPEC["stepsize"], dtype=float)  # g2 and alpha fixed
RPRS = 0.117
NDATA = 40
# Gaussian on kappa (index 0); Jeffreys on beta (index 4, bounds 0.55-1.4: log is defined everywhere)
PRIOR = np.array([-0.6, 0.0, 0.0, 0.0, 0.0, 0.0])
PRIORLOW = np.array([0.05, 0.0, 0.0, 0.0, -1.0, 0.0])


@pytest.fixture(scope="module")
def api(built):
    from bart_b200 import api as a
    a.lib()
    return a


def black_body_star(wn):
    starwn = np.linspace(wn[0] - 10, wn[-1] + 10, 3000)
    hc_k = 6.6260755e-27 * 2.99792458e10 / 1.380658e-16
    return starwn, 2 * 6.6260755e-27 * 2.99792458e10 ** 2 * starwn ** 3 / np.expm1(hc_k * starwn / 6300.0) * np.pi


@pytest.fixture(scope="module")
def retr(workdir):
    """The retr_tiny_eclipse set-up on a 30-layer atmosphere with 40 filters; data = the band
    oracle at the truth plus seeded 0.5 % noise, uncertainties 0.5 % of the data."""
    from bart_b200 import synth
    from oracle import retrieval_oracle as ro
    case = synth.make_case(os.path.join(workdir, "retr_scale40"), shape="tiny", solution="eclipse",
                           seed=SPEC["case"]["seed"], nlayer=30, nfilters=NDATA)
    starwn, starfl = black_body_star(case["wn"])
    conv = ro.Converter(case["press_bar"], case["species"], case["abund"], MOLFIT, "line",
                        pt_args=cases.W12_PTARGS)
    band = ro.BandOracle(case["cfg"], conv, case["filters"], starwn, starfl, RPRS)
    truth = band(SPEC["truth"])[0]
    data = truth * (1.0 + 0.005 * np.random.RandomState(4040).normal(size=truth.size))
    uncert = 0.005 * np.abs(data)
    assert data.size == NDATA and (data > 0).all()
    return dict(case=case, starwn=starwn, starfl=starfl, band=band, data=data, uncert=uncert)


def setup(api, retr):
    case = retr["case"]
    tr = api.Transit(case["cfg"])
    wn = tr.get_waveno_arr()
    tr.set_filters(*api.filters_from_files(wn, case["filters"], retr["starwn"], retr["starfl"]), RPRS)
    npars = tr.converter_init(case["press_bar"], case["species"], case["abund"], MOLFIT, "line",
                              pt_args=cases.W12_PTARGS, nrad=0)
    assert npars == len(PARAMS) and tr.nfilters == NDATA
    return tr


def test_bandflux_from_params_40_filters(api, retr):
    """parameters -> 40 band fluxes in one call against converter -> forward model -> band
    integration of the oracle; temperature-bound and abundance rejections come back as -1."""
    tr = setup(api, retr)
    rng = np.random.default_rng(40)
    params = np.repeat(np.array(SPEC["truth"])[None], 64, 0)
    params[:, STEPSIZE > 0] += rng.normal(0, 2, (64, 4)) * STEPSIZE[STEPSIZE > 0]
    params[40:56, :5] = rng.uniform(PMIN[:5], PMAX[:5], (16, 5))   # many outside 400-3000 K
    params[56:, 5] = 4.2                                           # CH4 10^4.2 x 1e-4: metals > 1
    bf, status = tr.bandflux_from_params(params)
    ref = retr["band"](params)
    _, ostatus, _ = retr["band"].conv.profiles(params)
    assert np.array_equal(status, ostatus)
    ok = status == 0
    assert ok.sum() >= 40 and (status == api.REJ_TBOUNDS).any() and (status == api.REJ_ABUND).any()
    assert np.all(bf[~ok] == -1.0) and np.all(ref[~ok] == -1.0)
    assert relerr(bf[ok], ref[ok]) < 1e-8
    tr.free_memory()


def test_demc_large_population_priors_fgamma_fepsilon(api, retr):
    """37 chains x 40 generations with both priors, fgamma 0.8 and fepsilon 0.02, against
    retrieval_oracle.demc on the same start points and streams."""
    from bart_b200 import driver
    from oracle import retrieval_oracle as ro
    nchains, chainsize = 37, 40
    ifree = np.where(STEPSIZE > 0)[0]
    rng = np.random.RandomState(37)
    p0 = np.repeat(PARAMS[None], nchains, 0)
    p0[:, ifree] += rng.normal(0, 3, (nchains, len(ifree))) * STEPSIZE[ifree]
    p0[[5, 20, 36], 4] = PMIN[4]                  # chains on a bound: proposals leave the box
    p0 = np.clip(p0, PMIN, PMAX)
    dr = driver.demc_draws(rng, nchains, chainsize, STEPSIZE[ifree])
    data, uncert = retr["data"], retr["uncert"]
    kw = dict(burnin=5, fgamma=0.8, fepsilon=0.02, draws=dr)
    tr = setup(api, retr)
    out = driver.run_demc(tr, data, uncert, p0, PMIN, PMAX, STEPSIZE, nchains * chainsize, nchains,
                          prior=PRIOR, priorlow=PRIORLOW, **kw)
    ref = ro.demc(retr["band"], data, uncert, p0, PMIN, PMAX, STEPSIZE, nchains * chainsize, nchains,
                  prior=PRIOR, priorlow=PRIORLOW, priorup=PRIORLOW, **kw)
    assert out["allparams"].shape == (nchains, len(ifree), chainsize)
    assert np.array_equal(out["allparams"], ref["allparams"])
    assert np.array_equal(out["params"], ref["params"])
    assert np.array_equal(out["numaccept"], ref["numaccept"])
    assert np.array_equal(out["outbounds"], ref["outbounds"])
    assert np.array_equal(out["bestp"], ref["bestp"])
    assert 0 < ref["numaccept"].sum() < nchains * (chainsize - 5) and ref["outbounds"].sum() > 0
    assert relerr(out["currchisq"], ref["currchisq"]) < 1e-6
    assert abs(out["bestchisq"] / ref["bestchisq"] - 1) < 1e-6
    assert relerr(out["bestmodel"], ref["bestmodel"]) < 1e-6
    assert np.array_equal(out["allmodel"] == 0, ref["allmodel"] == 0)
    assert relerr(out["allmodel"], ref["allmodel"]) < 1e-6
    # the same streams without priors: the priors decided at least one proposal
    plain = driver.run_demc(tr, data, uncert, p0, PMIN, PMAX, STEPSIZE, nchains * chainsize, nchains,
                            **kw)
    assert not np.array_equal(plain["allparams"], out["allparams"])
    tr.free_memory()


def test_snooker_long_run_regrows_history_across_grtest_segments(api, retr):
    """10 chains x 250 generations of walk='snooker' with both priors, grtest on: ten device calls
    between MC3's checkpoints, and the history outgrows its reservation twice on the way.  Against
    retrieval_oracle.snooker on the same seed, and against the one-call run."""
    from bart_b200 import driver
    from oracle import retrieval_oracle as ro
    nchains, numit, burnin, seed = 10, 2500, 10, 2500
    chainsize = numit // nchains
    # checkpoints every chainsize / 10 = 25 generations: calls of 25 generations each.  History
    # capacity (transit.cu snooker_reserve_rows: a request for r rows reserves r + r/2 + 16):
    #   init    hsize 11 + 64 = 75 -> 128 rows
    #   call k  needs 11 + 25 k + 1 rows: 37, 62, 87, 112, then 137 at call 5 -> 221 rows, the 111
    #           filled rows copied over; 162, 187, 212, then 237 at call 9 -> 371 rows, 211 copied;
    #           262 at call 10
    #   end     11 + 250 = 261 rows
    cuts = driver.gr_checkpoints(chainsize)
    assert cuts == list(range(24, chainsize, 25))
    data, uncert = retr["data"], retr["uncert"]
    kw = dict(prior=PRIOR, priorlow=PRIORLOW, burnin=burnin, thinning=1, fgamma=0.8, fepsilon=0.02)
    tr = setup(api, retr)
    np.random.seed(seed)
    out = driver.run_snooker(tr, data, uncert, PARAMS, PMIN, PMAX, STEPSIZE, numit, nchains,
                             grtest=True, **kw)
    np.random.seed(seed)
    ref = ro.snooker(retr["band"], data, uncert, PARAMS, PMIN, PMAX, STEPSIZE, numit, nchains,
                     priorup=PRIORLOW, **kw)
    assert ref["Zsize"] == 261 and out["Z"].shape == (261, nchains, len(PARAMS))
    assert np.array_equal(out["allparams"], ref["allparams"])
    assert np.array_equal(out["Z"], ref["Z"][:ref["Zsize"]])
    assert np.array_equal(out["numaccept"], ref["numaccept"])
    assert np.array_equal(out["outbounds"], ref["outbounds"])
    assert np.array_equal(out["bestp"], ref["bestp"])
    assert 0 < ref["numaccept"].sum() < nchains * (chainsize - burnin)
    assert relerr(out["Zchisq"], ref["Zchisq"][:ref["Zsize"]]) < 1e-6
    assert relerr(out["currchisq"], ref["currchisq"]) < 1e-6
    assert abs(out["bestchisq"] / ref["bestchisq"] - 1) < 1e-6
    assert [i for i, _ in out["psrf"]] == cuts
    for i, psrf in out["psrf"]:
        assert np.array_equal(psrf, driver.gelman_rubin(ref["allparams"][:, :, burnin:i + 1]), equal_nan=True)
    # one call (one regrowth, from the 11 initial rows): the same chains and history
    np.random.seed(seed)
    one = driver.run_snooker(tr, data, uncert, PARAMS, PMIN, PMAX, STEPSIZE, numit, nchains, **kw)
    assert one["psrf"] == []
    assert np.array_equal(one["allparams"], out["allparams"])
    assert np.array_equal(one["Z"], out["Z"])
    tr.free_memory()


def test_band_integration_filter_widths(api, get_case):
    """K4 over hand-built filters on the 2501-sample demo grid -- one trapezoid at either end of the
    spectrum, 2, 128, 511, 512, 513 and 1024 trapezoids (a pass is 512), the whole spectrum, 200
    random overlapping ones -- against oracle.bandflux, with and without a stellar spectrum."""
    from oracle import oracle as orc
    case, models, _ = get_case("demo_eclipse")
    tr = api.Transit(case["cfg"])
    wn = tr.get_waveno_arr()
    nw = len(wn)
    assert nw == 2501
    spectra, status = tr.run_batch(models)
    assert (status == 0).all()
    rng = np.random.default_rng(2501)
    fixed = [(0, 2), (nw - 2, 2), (7, 3), (100, 129), (640, 512), (1200, 513), (1713, 514),
             (nw - 1025, 1025), (0, nw)]
    count = np.concatenate([[c for _, c in fixed], rng.integers(2, 1400, 200)])
    start = np.concatenate([[s for s, _ in fixed], rng.integers(0, nw - count[len(fixed):] + 1)])
    assert (start + count <= nw).all()
    weight = [rng.uniform(0.05, 2.0, c) for c in count]
    star = [rng.uniform(0.5, 3.0, c) for c in count]
    filt = [(w, s, np.arange(a, a + c)) for w, s, a, c in zip(weight, star, start, count)]
    rprs = 0.12

    def check(bf, **kw):
        ref = np.array([orc.bandflux(sp, wn, filt, **kw) for sp in spectra])
        assert (ref > 0).all()
        err = np.max(np.abs(bf - ref) / ref, axis=0)
        assert not (err > 1e-12).any(), "filters of %s samples" % sorted(set(count[err > 1e-12]))

    tr.set_filters(start, count, np.concatenate(weight), np.concatenate(star), rprs)
    bf = tr.band_integrate(spectra)
    check(bf, star=True, rprs=rprs)
    bf2, status = tr.bandflux_batch(models)
    assert np.array_equal(bf2, bf) and (status == 0).all()
    tr.set_filters(start, count, np.concatenate(weight), None, 1.0)
    check(tr.band_integrate(spectra), star=False)
    tr.free_memory()
