"""CPU: the retrieval-loop oracle (oracle/retrieval_oracle.py) against golden vectors produced by
the reference's own Python code (tests/golden/make_golden_retrieval.py): code/PT.py, the
BARTfunc.py input converter, and a seeded run of the reference's MCcubed.mc.mcmc (DE-MC)."""
import os
import numpy as np
import pytest
import cases
from oracle import retrieval_oracle as ro

G = cases.GOLDEN_DIR


def test_expn2_and_pt_models_vs_reference():
    d = np.load(os.path.join(G, "retrieval_pt.npz"))
    e = ro.expn(2, d["x"])
    ok = d["expn2"] > 0
    assert np.max(np.abs(e[ok] - d["expn2"][ok]) / d["expn2"][ok]) < 1e-15
    assert np.all(e[~ok] == 0)
    p = d["pressure"]
    rstar, tstar, tint, sma, grav = d["ptargs"]
    for q, Tc, Tt in zip(d["pars"], d["T_const"], d["T_thorngren"]):
        assert np.max(np.abs(ro.PT_line(p, *q, rstar, tstar, tint, sma, grav) / Tc - 1)) < 1e-14
        assert np.max(np.abs(ro.PT_line(p, *q, rstar, tstar, tint, sma, grav, "thorngren") / Tt - 1)) < 1e-14
    for q, T in zip(d["apars"], d["T_adiabatic"]):
        assert np.array_equal(ro.PT_adiabatic(p, *q), T)


def test_system_parameters_from_tep_files():
    """driver.system_from_tep against the reference's reader.py + BARTfunc.py:157-172,204-211 on the
    two TEP files the reference ships."""
    from bart_b200 import driver
    g = np.load(os.path.join(G, "tep_systems.npz"))
    for name, fn in (("wasp12b", "WASP-12b.tep"), ("hd209458b", "HD209458b.tep")):
        s = driver.system_from_tep(os.path.join(G, "ref_inputs", fn), tint=100.0)
        got = np.array([s["tstar"], s["rstar"], s["sma"], s["rplanet"], s["mplanet"], s["gplanet"], s["rprs"]])
        assert np.array_equal(got, g[name]), (name, got, g[name])
        assert s["pt_args"] == (s["rstar"], s["tstar"], 100.0, s["sma"], s["gplanet"])


def test_smoothed_pt_models_vs_reference():
    """PT_NoInversion / PT_Inversion / PT_piette (incl. the restated scipy Gaussian filter and
    degree-1 spline) against code/PT.py on two pressure grids; the parameter sets PT.py refuses
    are refused."""
    g = np.load(os.path.join(G, "retrieval_pt_smooth.npz"))
    for tag in "ab":
        p = g["pressure_" + tag][::-1]
        for name, fn in (("noinv", ro.PT_NoInversion), ("inv", ro.PT_Inversion), ("piette", ro.PT_piette)):
            pars, T, phys = (g["%s_%s_%s" % (name, k, tag)] for k in ("pars", "T", "phys"))
            assert phys.sum() >= 30
            for q, Tref, ok in zip(pars, T, phys):
                try:
                    t = fn(p, *q)[::-1]
                except ro.NonPhysical:
                    assert not ok
                    continue
                assert ok and np.max(np.abs(t - Tref) / Tref) < 2e-15


def test_converter_rejects_refused_pt_parameters():
    g = np.load(os.path.join(G, "retrieval_pt_smooth.npz"))
    press = g["pressure_a"]
    nl = len(press)
    species = ["H2", "He", "H2O"]
    ab = np.tile([0.85, 0.149, 1e-3], (nl, 1))
    conv = ro.Converter(press, species, ab, ("H2O",), "madhu_noinv", tmin=0.0, tmax=1e9)
    pars = np.column_stack([g["noinv_pars_a"], np.zeros(len(g["noinv_pars_a"]))])
    prof, status, _ = conv.profiles(pars)
    assert np.array_equal(status == ro.REJ_PTMODEL, g["noinv_phys_a"] == 0) and (status == 0).sum() >= 30
    ok = status == 0
    assert np.max(np.abs(prof[ok, :nl] / g["noinv_T_a"][ok] - 1)) < 2e-15


@pytest.mark.parametrize("name", list(cases.RETRIEVAL))
def test_converter_vs_reference(name, workdir):
    case, spec, extra = cases.build_retrieval(name, workdir)
    d = np.load(os.path.join(G, "retrieval_conv_%s.npz" % name))
    conv = ro.Converter(case["press_bar"], case["species"], case["abund"], spec["molfit"], spec["pt"],
                        pt_args=extra["pt_args"], nrad=spec["nrad"], ncloud=spec["ncloud"],
                        nray=spec["nray"])
    prof, status, knobs = conv.profiles(d["params"])
    assert np.array_equal(status, d["status"])
    assert set(np.unique(status)) == {0, 16, 32}
    ok = status == 0
    assert np.max(np.abs(prof[ok] - d["profiles"][ok]) / np.abs(d["profiles"][ok])) < 1e-14
    c = conv.npt
    if spec["nrad"]:
        assert np.array_equal(knobs["refradius"], d["params"][:, c]); c += 1
    if spec["ncloud"]:
        assert np.array_equal(knobs["cloudtop"], d["params"][:, c]); c += 1
    if spec["nray"]:
        assert np.array_equal(knobs["scat_logext"], d["params"][:, c])


def test_converter_polar_scattering_takes_one_slot(workdir):
    """Polar scattering (nray = 2, `scattering = polar`) takes one parameter slot, like Lecavelier
    scattering, and leaves its value unused: molecule k's factor is parameter
    npt + nrad + ncloud + 1 + k."""
    case, spec, extra = cases.build_retrieval("retr_small4_transit", workdir)
    molfit = spec["molfit"]
    conv = ro.Converter(case["press_bar"], case["species"], case["abund"], molfit, "line",
                        pt_args=extra["pt_args"], nrad=1, ncloud=1, nray=2)
    nPT, nradfit, ncloud, nray = 5, 1, 1, 1          # BARTfunc counts the scattering parameter once
    nmolfit = len(molfit)
    assert conv.npars == nPT + nradfit + ncloud + nray + nmolfit == len(spec["params"])
    rng = np.random.default_rng(31)
    M = 24
    params = rng.uniform(spec["pmin"], spec["pmax"], (M, conv.npars))
    params[:, :nPT] = np.array(spec["params"][:nPT]) + rng.normal(0, 0.05, (M, nPT))
    params[:, -nmolfit:] = rng.uniform(-2.0, 1.0, (M, nmolfit))
    params[::5, -2] = 4.2                             # CO: metals past 1
    prof, status, knobs = conv.profiles(params)
    assert (status == 0).sum() >= 12 and (status == 32).any()
    # BARTfunc.py:333-347 on the converter's own temperatures (make_golden_retrieval.golden_converter)
    species = np.asarray(case["species"])
    abundances = case["abund"]
    iH2 = np.where(species == "H2")[0]
    iHe = np.where(species == "He")[0]
    ratio = (abundances[:, iH2] / abundances[:, iHe]).squeeze()
    imetals = np.where((species != "He") & (species != "H2") & (species != "H-") & (species != "e-"))[0]
    imol = [case["species"].index(m) for m in molfit]
    nl = len(case["press_bar"])
    for m in np.where(status == 0)[0]:
        par = params[m]
        aprofiles = abundances.T.copy()
        for i in np.arange(nmolfit):
            mm = imol[i]
            aprofiles[mm] = abundances[:, mm] * 10.0 ** par[nPT + nradfit + ncloud + nray + i]
        q = 1.0 - np.sum(aprofiles[imetals], axis=0)
        aprofiles[iH2] = ratio * q / (1.0 + ratio)
        aprofiles[iHe] = q / (1.0 + ratio)
        assert np.array_equal(prof[m, :nl], conv.temperature(par[:nPT]))
        assert np.array_equal(prof[m, nl:], aprofiles.ravel())
    assert np.array_equal(knobs["refradius"], params[:, nPT])
    assert np.array_equal(knobs["cloudtop"], params[:, nPT + 1])
    assert np.all(knobs["scat_flag"] == 2) and np.all(knobs["scat_logext"] == 0.0)
    # whatever the polar slot holds, the profiles are the same bit for bit
    for v in (-9.0, 3.0, np.nan):
        p2 = params.copy()
        p2[:, nPT + nradfit + ncloud] = v
        prof2, status2, knobs2 = conv.profiles(p2)
        assert np.array_equal(prof2, prof) and np.array_equal(status2, status)
        assert all(np.array_equal(knobs2[k], knobs[k]) for k in knobs)


@pytest.mark.parametrize("name", list(cases.RETRIEVAL))
def test_demc_oracle_reproduces_reference_mc3(name, built, workdir):
    """Same seed, same model function -> the reference's chain trace bit for bit."""
    case, spec, extra = cases.build_retrieval(name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    conv = ro.Converter(case["press_bar"], case["species"], case["abund"], spec["molfit"], spec["pt"],
                        pt_args=extra["pt_args"], nrad=spec["nrad"], ncloud=spec["ncloud"],
                        nray=spec["nray"])
    band = ro.BandOracle(case["cfg"], conv, case["filters"], extra["starwn"], extra["starfl"],
                         extra["rprs"])
    np.random.seed(spec["seed"])
    out = ro.demc(band, d["data"], d["uncert"], spec["params"], spec["pmin"], spec["pmax"],
                  spec["stepsize"], spec["numit"], spec["nchains"], burnin=spec["burnin"])
    assert np.array_equal(out["allparams"], d["allparams"])
    assert np.array_equal(out["bestp"], d["bestp"])
    # MC3's `savemodel` file (BART.cfg: band_eclipse.npy): models of the chains' current states,
    # zeros until a chain's first acceptance (mcmc.py:649-651)
    assert np.array_equal(out["allmodel"], d["allmodel"])
    assert (d["allmodel"][:, :, 0] == 0).all(axis=1).any()
    nacc = out["numaccept"].sum()
    assert 0 < nacc < spec["numit"]
    # the run resumed from its own savefile / savemodel (mcmc.py:254-269), new seed
    np.random.seed(spec["seed"] + 1)
    out2 = ro.demc(band, d["data"], d["uncert"], spec["params"], spec["pmin"], spec["pmax"],
                   spec["stepsize"], spec["numit"], spec["nchains"], burnin=spec["burnin"],
                   resume=(out["allparams"], out["allmodel"]))
    nold = d["allparams"].shape[2]
    assert d["resume_allparams"].shape[2] == 2 * nold
    assert np.array_equal(out2["allparams"], d["resume_allparams"])
    assert np.array_equal(out2["allmodel"], d["resume_allmodel"])
    assert np.array_equal(out2["bestp"], d["resume_bestp"])


@pytest.mark.parametrize("thinning", [1, 3])
@pytest.mark.parametrize("name", list(cases.RETRIEVAL))
def test_snooker_oracle_reproduces_reference_mc3(name, thinning, built, workdir):
    """walk='snooker' (the walk every BART example configures), MC3's MPI mode: same seed, same
    model function -> the reference's chain trace bit for bit."""
    case, spec, extra = cases.build_retrieval(name, workdir)
    d = np.load(os.path.join(G, "retrieval_snooker_%s_thin%d.npz" % (name, thinning)))
    conv = ro.Converter(case["press_bar"], case["species"], case["abund"], spec["molfit"], spec["pt"],
                        pt_args=extra["pt_args"], nrad=spec["nrad"], ncloud=spec["ncloud"],
                        nray=spec["nray"])
    band = ro.BandOracle(case["cfg"], conv, case["filters"], extra["starwn"], extra["starfl"],
                         extra["rprs"])
    np.random.seed(spec["seed"] + thinning)
    out = ro.snooker(band, d["data"], d["uncert"], spec["params"], spec["pmin"], spec["pmax"],
                     spec["stepsize"], spec["numit"], spec["nchains"], burnin=spec["burnin"],
                     thinning=thinning)
    assert np.array_equal(out["allparams"], d["allparams"])
    assert np.array_equal(out["bestp"], d["bestp"])
    assert np.array_equal(out["allmodel"], d["allmodel"])
    assert out["hsize"] == spec["nchains"] + 1
    assert out["Zsize"] == out["hsize"] + len(range(0, out["allparams"].shape[2], thinning))
    # the walk exercised projected snooker jumps and their Metropolis factor
    assert np.any(out["mrfactor"] != 1.0)
    nacc = out["numaccept"].sum()
    assert 0 < nacc < spec["numit"]


def test_gelman_rubin_matches_reference(built):
    """driver.gelman_rubin / gr_checkpoints against the reference's MCcubed/mc/gelman_rubin.py
    evaluated at MC3's own checkpoints (mcmc.py:238,663-686)."""
    from bart_b200 import driver
    g = np.load(os.path.join(G, "retrieval_gr.npz"))
    for name, spec in cases.RETRIEVAL.items():
        d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
        allp, burnin = d["allparams"], spec["burnin"]
        its = [i for i in driver.gr_checkpoints(allp.shape[2]) if i > burnin]
        assert its == list(g["its_" + name]) and len(its) >= 3
        for k, i in enumerate(its):
            assert np.allclose(driver.gelman_rubin(allp[:, :, burnin:i + 1]), g["psrf_" + name][k],
                               rtol=1e-12, atol=0, equal_nan=True)
    assert np.allclose(driver.gelman_rubin(g["conv_chains"][:, :, 50:300:2]), g["conv_psrf_thin2"], rtol=1e-12)
    assert np.all(g["conv_psrf_thin2"] < 1.01)


def test_run_segments_follows_mc3_convergence_logic():
    """The segment driver around the device-resident loop makes MC3's observable decisions
    (mcmc.py:662-690): PSRF at the checkpoints past burn-in, exit after two consecutive passes."""
    from bart_b200 import driver
    rng = np.random.RandomState(3)
    nch, nfree, chainsize, burnin, thinning = 6, 2, 200, 20, 1
    trace = rng.normal(0, 1, (nch, nfree, chainsize))
    trace[:, :, :60] += np.arange(nch)[:, None, None] * 3.0        # chains start far apart
    models = rng.normal(0, 1, (nch, 4, chainsize))
    state = {}

    def run(lo, hi):
        state["piece"] = (trace[:, :, lo:hi], models[:, :, lo:hi])

    # MC3's loop restated literally
    grflag, stop, hist = False, chainsize, []
    intsteps = chainsize / 10
    for i in range(chainsize):
        if ((i + 1) % intsteps == 0) and (i > 0) and i > burnin:
            psrf = driver.gelman_rubin(trace[:, :, burnin:i + 1:thinning])
            hist.append(i)
            if np.all(psrf < 1.01):
                if grflag:
                    stop = i + 1
                    break
                grflag = True
            else:
                grflag = False
    allp, allm, history, n = driver.run_segments(run, lambda: state["piece"], chainsize, burnin=burnin,
                                                 thinning=thinning, grtest=True, grexit=True)
    assert n == stop and [h[0] for h in history] == hist
    assert np.array_equal(allp, trace[:, :, :stop]) and np.array_equal(allm, models[:, :, :stop])
    # without grexit the whole chain runs and every checkpoint is reported; without grtest: one call
    allp2, _, history2, n2 = driver.run_segments(run, lambda: state["piece"], chainsize, burnin=burnin,
                                                 grtest=True, grexit=False)
    assert n2 == chainsize and np.array_equal(allp2, trace) and len(history2) >= len(history)
    calls = []
    driver.run_segments(lambda lo, hi: calls.append((lo, hi)) or run(lo, hi), lambda: state["piece"], chainsize)
    assert calls == [(0, chainsize)]


def test_energy_balance_oracle_vs_bartfunc_golden():
    """SURVEY 8 f2, third rejection test: oracle.retrieval_oracle.energy_balance against the
    statements of code/BARTfunc.py:366-383 executed verbatim with the reference's constants.py /
    reader.py on the shipped WASP-12b TEP file (tests/golden/ebalance.npz)."""
    import os
    import numpy as np
    from oracle import retrieval_oracle as ro
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ebalance.npz"))
    assert g["rejected"].sum() == 8 and len(g["rejected"]) == 16
    for m in range(len(g["rejected"])):
        e_in, e_out, rej = ro.energy_balance(g["spectra"][m], g["specwn"], float(g["tstar"]), float(g["rstar"]),
                                             float(g["sma"]), float(g["rplanet"]))
        assert abs(e_in / g["e_in"][m] - 1) < 1e-14
        assert abs(e_out / g["e_out"][m] - 1) < 1e-13
        assert rej == bool(g["rejected"][m])
