"""GPU: ensembles of independent retrievals in one device-resident MCMC loop
(bart_mcmc_init_ensemble, Transit.mcmc_init_ensemble, driver.run_demc_ensemble /
run_snooker_ensemble).  Every retrieval of an ensemble must come out bit-identical to the same
retrieval run alone on the same data, start points and random streams; an ensemble of one is the
lone retrieval byte for byte.

The lone runs evaluate a population of nchains models per generation, the ensemble one of
R x nchains; the eclipse kernel family depends on the batch size (the scan kernel of small batches
agrees with the other two to ~1e-10 only), so the ensemble-against-lone comparisons pin it with
BART_ECL_SMALL=0 for both runs."""
import os
import subprocess
import sys

import numpy as np
import pytest

import cases
from util import relerr

pytestmark = pytest.mark.gpu
G = cases.GOLDEN_DIR
HERE = os.path.dirname(os.path.abspath(__file__))
DEMC_KEYS = ("allparams", "allmodel", "params", "numaccept", "outbounds", "bestp", "bestchisq",
             "bestmodel", "currchisq", "models")
SNOOKER_KEYS = DEMC_KEYS + ("Z", "Zchisq")


@pytest.fixture(scope="module")
def api(built):
    from bart_b200 import api as a
    a.lib()
    return a


def setup(api, name, workdir):
    case, spec, extra = cases.build_retrieval(name, workdir)
    tr = api.Transit(case["cfg"])
    wn = tr.get_waveno_arr()
    start, count, weight, star = api.filters_from_files(wn, case["filters"], extra["starwn"], extra["starfl"])
    tr.set_filters(start, count, weight, star, extra["rprs"])
    tr.converter_init(case["press_bar"], case["species"], case["abund"], spec["molfit"], spec["pt"],
                      pt_args=extra["pt_args"], nrad=spec["nrad"], ncloud=spec["ncloud"],
                      nray=spec["nray"])
    return case, spec, extra, tr


def band_oracle(case, spec, extra):
    from oracle import retrieval_oracle as ro
    conv = ro.Converter(case["press_bar"], case["species"], case["abund"], spec["molfit"], spec["pt"],
                        pt_args=extra["pt_args"], nrad=spec["nrad"], ncloud=spec["ncloud"],
                        nray=spec["nray"])
    return ro.BandOracle(case["cfg"], conv, case["filters"], extra["starwn"], extra["starfl"],
                         extra["rprs"])


def same(a, b, keys):
    for k in keys:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.shape == y.shape and np.array_equal(x, y, equal_nan=True), k
    assert len(a["psrf"]) == len(b["psrf"])
    for (i, p), (j, q) in zip(a["psrf"], b["psrf"]):
        assert i == j and np.array_equal(p, q, equal_nan=True)


def ensemble_inputs(tr, spec, d, nretr, seed, reject_in=None):
    """Per retrieval: data (retrieval 0 the golden data, the others with seeded 1 % noise), start
    points scattered by RandomState(seed + r) like mcmc.py:296-306, and that RandomState for the
    random streams.  `reject_in`: a retrieval whose chains 1 and 2 start where the converter
    rejects the temperature profile."""
    from bart_b200 import driver
    nch = spec["nchains"]
    pmin, pmax, stepsize = (np.array(spec[k], dtype=float) for k in ("pmin", "pmax", "stepsize"))
    data, uncert, starts, rngs = [], [], [], []
    for r in range(nretr):
        noise = np.random.RandomState(900 + r).normal(size=len(d["data"]))
        data.append(d["data"] * (1 + 0.01 * noise) if r else d["data"])
        uncert.append(d["uncert"])
        rng = np.random.RandomState(seed + r)
        starts.append(driver.start_points(spec["params"], nch, stepsize, pmin, pmax, rng))
        rngs.append(rng)
    if reject_in is not None:
        cand = np.repeat(np.array(spec["params"], dtype=float)[None], 256, 0)
        cand[:, :5] = np.random.RandomState(77).uniform(pmin[:5], pmax[:5], (256, 5))
        _, status, _ = tr.profiles_from_params(cand)
        hot = cand[status == 16]
        assert len(hot) >= 2
        starts[reject_in][1:3] = hot[:2]
    return np.array(data), np.array(uncert), starts, rngs


@pytest.mark.parametrize("walk", ["demc", "snooker"])
@pytest.mark.parametrize("graph", ["1", "0"])
@pytest.mark.parametrize("name", list(cases.RETRIEVAL))
def test_ensemble_of_one_is_the_lone_retrieval(name, graph, walk, api, workdir, monkeypatch):
    """mcmc_init_ensemble with R = 1 == mcmc_init byte for byte, default kernel selection."""
    from bart_b200 import driver
    monkeypatch.setenv("BART_MCMC_GRAPH", graph)
    case, spec, extra, tr = setup(api, name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    nch, numit = spec["nchains"], spec["numit"]
    args = (spec["pmin"], spec["pmax"], spec["stepsize"], numit, nch)
    kw = dict(burnin=spec["burnin"])
    if walk == "demc":
        np.random.seed(spec["seed"])
        lone = driver.run_demc(tr, d["data"], d["uncert"], spec["params"], *args, **kw)
        ens = driver.run_demc_ensemble(tr, d["data"][None], d["uncert"][None], [spec["params"]], *args,
                                       rngs=[np.random.RandomState(spec["seed"])], **kw)
        keys = DEMC_KEYS
    else:
        np.random.seed(spec["seed"] + 3)
        lone = driver.run_snooker(tr, d["data"], d["uncert"], spec["params"], *args, thinning=3, **kw)
        ens = driver.run_snooker_ensemble(tr, d["data"][None], d["uncert"][None], [spec["params"]],
                                          *args, thinning=3,
                                          rngs=[np.random.RandomState(spec["seed"] + 3)], **kw)
        keys = SNOOKER_KEYS
    assert api.lib().bart_mcmc_nretr() == 1 and len(ens) == 1
    same(ens[0], lone, keys + ("allstack",))
    assert tr.mcmc_get("params").shape == (1, nch, len(spec["params"]))
    assert tr.mcmc_get("bestchisq").shape == (1,)
    tr.free_memory()


@pytest.mark.parametrize("graph", ["1", "0"])
@pytest.mark.parametrize("name", list(cases.RETRIEVAL))
def test_demc_ensemble_equals_lone_runs(name, graph, api, workdir, monkeypatch):
    """R = 4: every retrieval equals run_demc of that retrieval alone on the same streams, one of
    them with chains starting in the temperature-rejection region; retrieval 0 (the golden data)
    also matches the oracle's DE-MC."""
    from bart_b200 import driver
    from oracle import retrieval_oracle as ro
    monkeypatch.setenv("BART_MCMC_GRAPH", graph)
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    case, spec, extra, tr = setup(api, name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    nch, numit, R = spec["nchains"], spec["numit"], 4
    stepsize = np.array(spec["stepsize"], dtype=float)
    data, uncert, starts, rngs = ensemble_inputs(tr, spec, d, R, spec["seed"], reject_in=2)
    chainsize = int(np.ceil(numit / nch))
    draws = [driver.demc_draws(rngs[r], nch, chainsize, stepsize[stepsize > 0]) for r in range(R)]
    args = (spec["pmin"], spec["pmax"], stepsize, numit, nch)
    kw = dict(burnin=spec["burnin"])
    ens = driver.run_demc_ensemble(tr, data, uncert, starts, *args, draws=draws, **kw)
    assert api.lib().bart_mcmc_nretr() == R
    for r in range(R):
        lone = driver.run_demc(tr, data[r], uncert[r], starts[r], *args, draws=draws[r], **kw)
        same(ens[r], lone, DEMC_KEYS + ("allstack",))
    assert not np.array_equal(ens[0]["allparams"], ens[1]["allparams"])
    ref = ro.demc(band_oracle(case, spec, extra), data[0], uncert[0], starts[0], *args, draws=draws[0], **kw)
    assert np.array_equal(ens[0]["numaccept"], ref["numaccept"])
    assert np.array_equal(ens[0]["params"], ref["params"])
    assert np.array_equal(ens[0]["outbounds"], ref["outbounds"])
    tr.free_memory()


@pytest.mark.parametrize("graph", ["1", "0"])
@pytest.mark.parametrize("thinning", [1, 3])
@pytest.mark.parametrize("name", list(cases.RETRIEVAL))
def test_snooker_ensemble_equals_lone_runs(name, thinning, graph, api, workdir, monkeypatch):
    from bart_b200 import driver
    monkeypatch.setenv("BART_MCMC_GRAPH", graph)
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    case, spec, extra, tr = setup(api, name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    nch, numit, R = spec["nchains"], spec["numit"], 3
    pmin, pmax, stepsize = (np.array(spec[k], dtype=float) for k in ("pmin", "pmax", "stepsize"))
    ifree = stepsize > 0
    data, uncert, starts, rngs = ensemble_inputs(tr, spec, d, R, spec["seed"] + thinning, reject_in=1)
    chainsize, hsize = int(np.ceil(numit / nch)), nch + 1
    draws = [driver.snooker_draws(rngs[r], nch, int(ifree.sum()), chainsize, hsize, thinning,
                                  stepsize[ifree], pmin[ifree], pmax[ifree]) for r in range(R)]
    args = (pmin, pmax, stepsize, numit, nch)
    kw = dict(burnin=spec["burnin"], thinning=thinning, hsize=hsize)
    ens = driver.run_snooker_ensemble(tr, data, uncert, starts, *args, draws=draws, **kw)
    assert sum(len(dr["usnooker"]) for dr in draws) > 0
    for r in range(R):
        lone = driver.run_snooker(tr, data[r], uncert[r], starts[r], *args, draws=draws[r], **kw)
        same(ens[r], lone, SNOOKER_KEYS + ("allstack",))
    assert not np.array_equal(ens[0]["Z"], ens[2]["Z"])
    tr.free_memory()


def test_snooker_ensemble_long_run_history_regrowth_and_grtest(api, workdir, monkeypatch):
    """250 generations with grtest: ten device calls between MC3's checkpoints, and the shared
    history outgrows its reservation on the way (7 initial rows + 250); each retrieval's PSRF
    history equals driver.gelman_rubin on its lone trace."""
    from bart_b200 import driver
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    name = "retr_tiny_eclipse"
    case, spec, extra, tr = setup(api, name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    nch, R, chainsize, burnin = spec["nchains"], 3, 250, 10
    data, uncert, _, _ = ensemble_inputs(tr, spec, d, R, 0)
    args = (spec["pmin"], spec["pmax"], spec["stepsize"], chainsize * nch, nch)
    kw = dict(burnin=burnin, thinning=1, grtest=True)
    # start points scattered and streams drawn by each retrieval's own rng
    ens = driver.run_snooker_ensemble(tr, data, uncert, [spec["params"]] * R, *args,
                                      rngs=[np.random.RandomState(4242 + r) for r in range(R)], **kw)
    cuts = driver.gr_checkpoints(chainsize)
    for r in range(R):
        lone = driver.run_snooker(tr, data[r], uncert[r], spec["params"], *args,
                                  rng=np.random.RandomState(4242 + r), **kw)
        same(ens[r], lone, SNOOKER_KEYS)
        assert ens[r]["Z"].shape[0] == nch + 1 + chainsize
        assert [i for i, _ in ens[r]["psrf"]] == cuts
        for i, psrf in ens[r]["psrf"]:
            assert np.array_equal(psrf, driver.gelman_rubin(lone["allparams"][:, :, burnin:i + 1]),
                                  equal_nan=True)
    tr.free_memory()


# ---- production size: the 40-filter, 37-chain configuration of test_gpu_retrieval_scale.py ----
SPEC = cases.RETRIEVAL["retr_tiny_eclipse"]
PARAMS, PMIN, PMAX = (np.array(SPEC[k], dtype=float) for k in ("params", "pmin", "pmax"))
STEPSIZE = np.array(SPEC["stepsize"], dtype=float)
PRIOR = np.array([-0.6, 0.0, 0.0, 0.0, 0.0, 0.0])
PRIORLOW = np.array([0.05, 0.0, 0.0, 0.0, -1.0, 0.0])
NDATA, RPRS = 40, 0.117


@pytest.fixture(scope="module")
def retr40(workdir):
    from bart_b200 import synth
    from oracle import retrieval_oracle as ro
    case = synth.make_case(os.path.join(workdir, "ens_scale40"), shape="tiny", solution="eclipse",
                           seed=SPEC["case"]["seed"], nlayer=30, nfilters=NDATA)
    wn = case["wn"]
    starwn = np.linspace(wn[0] - 10, wn[-1] + 10, 3000)
    hc_k = 6.6260755e-27 * 2.99792458e10 / 1.380658e-16
    starfl = 2 * 6.6260755e-27 * 2.99792458e10 ** 2 * starwn ** 3 / np.expm1(hc_k * starwn / 6300.0) * np.pi
    conv = ro.Converter(case["press_bar"], case["species"], case["abund"], SPEC["molfit"], "line",
                        pt_args=cases.W12_PTARGS)
    band = ro.BandOracle(case["cfg"], conv, case["filters"], starwn, starfl, RPRS)
    truth = band(SPEC["truth"])[0]
    return dict(case=case, starwn=starwn, starfl=starfl, band=band, truth=truth)


def test_demc_ensemble_production_size(api, retr40, monkeypatch):
    """R = 8 retrievals x 37 chains (296 models per generation: the throughput eclipse kernel, one
    chi-squared CTA per retrieval), 40 data points, both priors, fgamma 0.8, fepsilon 0.02: every
    retrieval equals its lone run, retrieval 0 equals the oracle's DE-MC."""
    from bart_b200 import driver
    from oracle import retrieval_oracle as ro
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    case = retr40["case"]
    tr = api.Transit(case["cfg"])
    wn = tr.get_waveno_arr()
    tr.set_filters(*api.filters_from_files(wn, case["filters"], retr40["starwn"], retr40["starfl"]), RPRS)
    tr.converter_init(case["press_bar"], case["species"], case["abund"], SPEC["molfit"], "line",
                      pt_args=cases.W12_PTARGS, nrad=0)
    R, nch, chainsize = 8, 37, 24
    ifree = np.where(STEPSIZE > 0)[0]
    data, uncert, starts, draws = [], [], [], []
    for r in range(R):
        rng = np.random.RandomState(3700 + r)
        dat = retr40["truth"] * (1.0 + 0.005 * rng.normal(size=NDATA))
        data.append(dat); uncert.append(0.005 * np.abs(dat))
        p0 = np.repeat(PARAMS[None], nch, 0)
        p0[:, ifree] += rng.normal(0, 3, (nch, len(ifree))) * STEPSIZE[ifree]
        p0[[5, 20, 36], 4] = PMIN[4]
        starts.append(np.clip(p0, PMIN, PMAX))
        draws.append(driver.demc_draws(rng, nch, chainsize, STEPSIZE[ifree]))
    data, uncert = np.array(data), np.array(uncert)
    args = (PMIN, PMAX, STEPSIZE, nch * chainsize, nch)
    kw = dict(prior=PRIOR, priorlow=PRIORLOW, burnin=5, fgamma=0.8, fepsilon=0.02)
    ens = driver.run_demc_ensemble(tr, data, uncert, starts, *args, draws=draws, **kw)
    for r in range(R):
        lone = driver.run_demc(tr, data[r], uncert[r], starts[r], *args, draws=draws[r], **kw)
        same(ens[r], lone, DEMC_KEYS)
    ref = ro.demc(retr40["band"], data[0], uncert[0], starts[0], *args, priorup=PRIORLOW,
                  draws=draws[0], **kw)
    for k in ("allparams", "params", "numaccept", "outbounds", "bestp"):
        assert np.array_equal(ens[0][k], ref[k]), k
    assert 0 < ref["numaccept"].sum() and ref["outbounds"].sum() > 0
    assert relerr(ens[0]["currchisq"], ref["currchisq"]) < 1e-6
    assert abs(ens[0]["bestchisq"] / ref["bestchisq"] - 1) < 1e-6
    tr.free_memory()


def test_ensemble_continuation_and_resume(api, workdir, monkeypatch):
    """Two mcmc_run calls of n/2 generations == one call of n for an ensemble; mcmc_resume of an
    ensemble (nold, curmodel[R][C][D]) == each retrieval's lone resumed run."""
    from bart_b200 import driver
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    name = "retr_tiny_eclipse"
    case, spec, extra, tr = setup(api, name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    nch, R, n = spec["nchains"], 3, 16
    stepsize = np.array(spec["stepsize"], dtype=float)
    data, uncert, starts, rngs = ensemble_inputs(tr, spec, d, R, 55)
    draws = [driver.demc_draws(rngs[r], nch, n, stepsize[stepsize > 0]) for r in range(R)]
    starts = np.array(starts)
    init = lambda: tr.mcmc_init_ensemble(starts, spec["pmin"], spec["pmax"], stepsize, data, uncert,
                                         burnin=3)
    init()
    tr.mcmc_run(*driver.stack_demc_draws(draws, 0, n))
    one = {k: tr.mcmc_get(k) for k in ("allparams", "allmodel", "params", "numaccept", "bestp")}
    init()
    halves = []
    for h in (slice(0, n // 2), slice(n // 2, n)):
        tr.mcmc_run(*driver.stack_demc_draws(draws, h.start, h.stop))
        halves.append((tr.mcmc_get("allparams"), tr.mcmc_get("allmodel")))
    assert np.array_equal(np.concatenate([p for p, _ in halves], axis=3), one["allparams"])
    assert np.array_equal(np.concatenate([m for _, m in halves], axis=3), one["allmodel"])
    for k in ("params", "numaccept", "bestp"):
        assert np.array_equal(tr.mcmc_get(k), one[k]), k
    # resume from the last states and models of that run
    last = one["params"]
    curmodel = one["allmodel"][..., -1]
    rdraws = [driver.demc_draws(np.random.RandomState(66 + r), nch, n, stepsize[stepsize > 0]) for r in range(R)]
    tr.mcmc_init_ensemble(last, spec["pmin"], spec["pmax"], stepsize, data, uncert, burnin=20)
    tr.mcmc_resume(n, curmodel)
    tr.mcmc_run(*driver.stack_demc_draws(rdraws, 0, n))
    ens = {k: tr.mcmc_get(k) for k in ("allparams", "allmodel", "params", "numaccept", "bestp", "bestchisq")}
    for r in range(R):
        tr.mcmc_init(last[r], spec["pmin"], spec["pmax"], stepsize, data[r], uncert[r], burnin=20)
        tr.mcmc_resume(n, curmodel[r])
        dr = rdraws[r]
        tr.mcmc_run(dr["support"], dr["r1"], dr["r2"], dr["unif"], dr["ugamma"])
        for k in ("allparams", "allmodel", "params", "numaccept", "bestp"):
            assert np.array_equal(ens[k][r], tr.mcmc_get(k)), k
        assert ens["bestchisq"][r] == tr.mcmc_get("bestchisq")[0]
    assert ens["numaccept"].sum() > 0
    tr.free_memory()


def test_ensemble_refusals(api, workdir):
    """Wrong leading dimension, an r1 index out of range in retrieval 2, a usn_offset count
    mismatch, grexit=True and nretr = 0 are refused with a clear error."""
    from bart_b200 import driver
    name = "retr_tiny_eclipse"
    case, spec, extra, tr = setup(api, name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    nch, R, n = spec["nchains"], 3, 6
    pmin, pmax, stepsize = (np.array(spec[k], dtype=float) for k in ("pmin", "pmax", "stepsize"))
    ifree = stepsize > 0
    data, uncert, starts, rngs = ensemble_inputs(tr, spec, d, R, 99)
    draws = [driver.demc_draws(rngs[r], nch, n, stepsize[ifree]) for r in range(R)]
    tr.mcmc_init_ensemble(np.array(starts), pmin, pmax, stepsize, data, uncert)
    streams = driver.stack_demc_draws(draws, 0, n)
    with pytest.raises(api.BartError, match="3 retrievals"):
        tr.mcmc_run(*(s[:2] for s in streams))
    with pytest.raises(api.BartError, match="curmodel"):
        tr.mcmc_resume(0, np.zeros((nch, len(d["data"]))))
    bad = [s.copy() for s in streams]
    bad[1][2, 4, 3] = nch                              # r1 of retrieval 2, chain 4, generation 3
    with pytest.raises(api.BartError, match="retrieval 2, generation 3, chain 4"):
        tr.mcmc_run(*bad)
    tr.mcmc_run(*streams)                              # the loop is still usable
    # snooker: one generation's factor rows miscounted
    hsize = nch + 1
    sd = [driver.snooker_draws(np.random.RandomState(7 + r), nch, int(ifree.sum()), n, hsize, 1,
                               stepsize[ifree], pmin[ifree], pmax[ifree]) for r in range(R)]
    tr.mcmc_init_ensemble(np.array(starts), pmin, pmax, stepsize, data, uncert)
    with pytest.raises(api.BartError, match="z0"):
        tr.mcmc_snooker_init(sd[0]["z0"])
    tr.mcmc_snooker_init(np.stack([s["z0"] for s in sd]))
    snk = list(driver.stack_snooker_draws(sd, 0, n))
    ug = snk[8]
    ug[:, 2, 1] = np.where(ug[:, 2, 1] >= 0.1, 0.05, 0.5)          # counts no longer match
    with pytest.raises(api.BartError, match="usn_offset: retrieval 0, generation 2"):
        tr.mcmc_run_snooker(*snk)
    with pytest.raises(ValueError, match="grexit"):
        driver.run_demc_ensemble(tr, data, uncert, starts, pmin, pmax, stepsize, n * nch, nch,
                                 draws=draws, grtest=True, grexit=True)
    with pytest.raises(ValueError, match="grexit"):
        driver.run_snooker_ensemble(tr, data, uncert, starts, pmin, pmax, stepsize, n * nch, nch,
                                    draws=sd, grtest=True, grexit=True)
    with pytest.raises(api.BartError, match="0 retrievals"):
        tr.mcmc_init_ensemble(np.zeros((0, nch, len(pmin))), pmin, pmax, stepsize,
                              np.zeros((0, len(d["data"]))), np.zeros((0, len(d["data"]))))
    tr.free_memory()


# ---- host side of the ensemble drivers (no device work) ----
def test_grexit_and_mismatched_inputs_are_refused():
    from bart_b200 import driver
    kw = dict(pmin=[0.0], pmax=[1.0], stepsize=[0.1], numit=30, nchains=3)
    with pytest.raises(ValueError, match="grexit"):
        driver.run_demc_ensemble(None, np.zeros((2, 4)), np.ones((2, 4)), [[0.5]] * 2, grtest=True,
                                 grexit=True, **kw)
    with pytest.raises(ValueError, match="one entry per retrieval"):
        driver.run_demc_ensemble(None, np.zeros((2, 4)), np.ones((2, 4)), [[0.5]] * 3, **kw)
    with pytest.raises(ValueError, match="rngs needs one entry"):
        driver.run_demc_ensemble(None, np.zeros((2, 4)), np.ones((2, 4)), [[0.5]] * 2,
                                 rngs=[np.random.RandomState(0)], **kw)
    with pytest.raises(ValueError, match="retrieval 0 needs an rng"):
        driver.run_demc_ensemble(None, np.zeros((2, 4)), np.ones((2, 4)), [[0.5]] * 2, **kw)


def test_segment_bound_at_64_retrievals():
    """R = 64, 10 chains, 9 free parameters, 40 data points, 1e5 generations: one device call's
    streams and traces stay under ENSEMBLE_CALL_BYTES, not the 4.6 GB `support` alone would take."""
    from bart_b200 import driver
    R, C, F, D, n = 64, 10, 9, 40, 100000
    cap = driver._segment_cap(R, C, F, D)
    assert 1 <= cap < n
    assert R * C * cap * (8 * (F + 2 + F + D) + 2 * 4) <= driver.ENSEMBLE_CALL_BYTES
    assert driver._segment_cap(1, 3, 1, 1) > 1000


def test_run_segments_bounds_calls_and_keeps_psrf_per_retrieval():
    from bart_b200 import driver
    rng = np.random.RandomState(3)
    R, C, F, n = 3, 4, 2, 50
    trace = rng.normal(size=(R, C, F, n))
    calls = []

    def run(lo, hi):
        calls.append((lo, hi))

    def fetch():
        lo, hi = calls[-1]
        return trace[..., lo:hi], trace[..., lo:hi] * 2
    allp, allm, hist, chainlen = driver.run_segments(run, fetch, n, burnin=2, grtest=True, max_segment=7)
    assert max(hi - lo for lo, hi in calls) <= 7 and calls[0][0] == 0 and calls[-1][1] == n
    assert np.array_equal(allp, trace) and np.array_equal(allm, 2 * trace) and chainlen == n
    assert [i for i, _ in hist] == driver.gr_checkpoints(n)
    for i, psrf in hist:
        assert psrf.shape == (R, F)
        for r in range(R):
            assert np.array_equal(psrf[r], driver.gelman_rubin(trace[r, :, :, 2:i + 1]), equal_nan=True)


def test_stacked_snooker_offsets_are_absolute_rows():
    from bart_b200 import driver
    sd = [driver.snooker_draws(np.random.RandomState(r), 4, 2, 12, 5, 1, np.full(2, 0.1), np.zeros(2),
                               np.ones(2)) for r in range(3)]
    for d in sd:
        d["ugamma"][:, ::2] *= 0.1                                 # snooker jumps in most generations
    lo, hi = 3, 9
    snk = driver.stack_snooker_draws(sd, lo, hi)
    usn, off = snk[5], snk[6]
    assert off.shape == (3, hi - lo + 1) and off[0, 0] == 0 and off[-1, -1] == len(usn)
    for r, d in enumerate(sd):
        o = d["usn_offset"]
        assert np.array_equal(usn[off[r, 0]:off[r, -1]], d["usnooker"][o[lo]:o[hi]])
        assert np.array_equal(np.diff(off[r]), np.diff(o[lo:hi + 1]))
        assert np.array_equal(snk[0][r], d["support"][lo:hi]) and np.array_equal(snk[8][r], d["ugamma"][lo:hi])


def ngpus():
    try:
        out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=30).stdout
        return sum(1 for l in out.splitlines() if l.startswith("GPU "))
    except Exception:
        return 0


@pytest.mark.skipif(ngpus() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("p2p", [1, 0])
def test_two_rank_ensemble_equals_single_gpu(p2p, api, workdir, monkeypatch):
    """R = 4 with the flattened population (24 models) split over 2 ranks, through the fused
    peer-window all-gather and through NCCL: every rank's output equals the single-GPU ensemble."""
    wd = os.path.join(workdir, "ens_mr_%d" % p2p)
    os.makedirs(wd, exist_ok=True)
    env = dict(os.environ, BART_P2P=str(p2p), BART_ECL_SMALL="0")
    env.pop("LOCAL_RANK", None)
    outs = [os.path.join(wd, "out%d.npz" % r) for r in range(2)]
    procs = [subprocess.Popen([sys.executable, os.path.join(HERE, "ensemble_rank_worker.py"), str(r), "2",
                               wd, outs[r]], env=env, stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    logs = []
    for p in procs:
        try:
            o, _ = p.communicate(timeout=300)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise AssertionError("ensemble worker timed out")
        logs.append(o)
    for p, o in zip(procs, logs):
        assert p.returncode == 0, o[-3000:]
    res = [np.load(o) for o in outs]
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    sys.path.insert(0, HERE)
    import ensemble_rank_worker as w
    single = w.run_ensemble(api, os.path.join(wd, "single"), device=0)
    for r in res:
        if p2p:
            assert int(r["p2p"]) == 1, "peer windows were not mapped"
        for k in single:
            assert np.array_equal(r[k], single[k]), k
