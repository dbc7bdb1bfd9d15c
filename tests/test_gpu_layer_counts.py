"""GPU: layer counts past the ones the parity cases use, against the oracle (oracle/transit_oracle.c
and oracle/retrieval_oracle.py, both free of layer limits).

The column kernels stage a model's whole table in the shared memory of one block, so the layer
count picks the kernel: the transit tensor-core (DMMA) kernel runs two CTAs per SM up to 112 layers
and one up to ~220, the DFMA tile kernel takes over up to ~240, and past the last kernel that fits,
transit_init refuses the configuration and names the limit.  The input converter makes more than
one pass over the layers past 128 and stops staging its arrays in shared memory past 512 layers
(10 species)."""
import os
import re

import numpy as np
import pytest

import cases
from util import relerr, apply_setters

pytestmark = pytest.mark.gpu
TIGHT = 1e-8
# the per-model knobs of small4_transit_cloud
SETTERS = {"radius": 94500.0, "cloudtop": -2.0, "scattering": 0.5}
# few grid temperatures keep the opacity files of the deep cases small (400 ... 3000 K)
TEMPDELT = 650.0


@pytest.fixture(scope="module")
def api(built):
    from bart_b200 import api as a
    info = a.device_info()
    assert info["cc"][0] >= 10, info
    return a


def make(workdir, shape, solution, nlayer, tempdelt=TEMPDELT):
    from bart_b200 import synth
    name = "%s_%s_%d_t%g" % (shape, solution, nlayer, tempdelt)
    return synth.make_case(os.path.join(workdir, name), shape=shape, solution=solution,
                           seed=4000 + nlayer, nlayer=nlayer, tempdelt=tempdelt,
                           refradius_km=95000.0 if solution == "transit" else 123820.0)


def models_of(case, seed):
    from bart_b200 import synth
    molfit = ("CH4",) if len(case["shape"]["mols"]) == 1 else ("H2O", "CO2", "CO", "CH4")
    return synth.make_models(case, 2, seed=seed, molfit=molfit)


def layer_limit(api, cfg):
    """The configuration is refused by transit_init; -> the largest layer count the message names."""
    with pytest.raises(api.BartError) as e:
        api.Transit(cfg)
    m = re.search(r"supports at most (\d+) layers", str(e.value))
    assert m, str(e.value)
    return int(m.group(1))


def check_transit(api, case, models, monkeypatch):
    """Spectra of the default kernel choice and of the forced DFMA tile kernel within TIGHT of the
    oracle, last[] of the introspection kernel identical to the oracle's, nothing rejected.
    -> (default spectra, tile-kernel spectra)."""
    from oracle import oracle as orc
    tr = api.Transit(case["cfg"])
    apply_setters(tr, SETTERS)
    O = orc.Oracle(case["cfg"])
    apply_setters(O, SETTERS)
    assert tr.nlayer == case["nlayer"]
    ref = [O.run(models[m], inter=True) for m in range(models.shape[0])]
    tr.debug_keep(True)
    keep, status = tr.run_batch(models)
    assert (status == 0).all()
    for m, o in enumerate(ref):
        assert np.array_equal(tr.debug_get("last", m).astype(np.int64), o["last"])
        assert relerr(keep[m], o["spectrum"]) < TIGHT
    tr.debug_keep(False)
    out = []
    for mma in (None, "0"):
        if mma is None:
            monkeypatch.delenv("BART_TRANSIT_MMA", raising=False)
        else:
            monkeypatch.setenv("BART_TRANSIT_MMA", mma)
        spectra, status = tr.run_batch(models)
        assert (status == 0).all()
        for m, o in enumerate(ref):
            assert relerr(spectra[m], o["spectrum"]) < TIGHT, (mma, m)
        out.append(spectra)
    monkeypatch.delenv("BART_TRANSIT_MMA", raising=False)
    tr.free_memory()
    return out


# (shape, layers, above the DMMA kernel's limit): the DMMA kernel is chosen while its shared memory
# (kernels.cu transit_mma_smem) is at most 200 KB -- up to 224 layers for `tiny` (1 molecule, 1 CIA
# table), 213 for `small4` (4 molecules); 112 / 113 is its edge between two CTAs per SM and one.
# The tile kernel then runs `tiny` up to 244 layers: at 245 its 232 288 bytes of dynamic shared
# memory and 256 static ones exceed the 227 KB a block can have on a B200.
TRANSIT_COUNTS = [("tiny", 112, False), ("tiny", 113, False), ("tiny", 208, False),
                  ("tiny", 224, False), ("tiny", 225, True), ("tiny", 244, True),
                  ("small4", 213, False), ("small4", 214, True)]


@pytest.mark.parametrize("shape,nlayer,tile_only", TRANSIT_COUNTS)
def test_transit_across_the_kernel_boundaries(shape, nlayer, tile_only, api, workdir, monkeypatch):
    case = make(workdir, shape, "transit", nlayer)
    default, tile = check_transit(api, case, models_of(case, 500 + nlayer), monkeypatch)
    if tile_only:
        # past the DMMA kernel's limit the default choice is the tile kernel's production build
        assert np.array_equal(default, tile)


@pytest.mark.parametrize("shape", ["tiny", "small4"])
def test_transit_layer_limit_is_refused_at_init(shape, api, workdir, monkeypatch):
    L = layer_limit(api, make(workdir, shape, "transit", 321)["cfg"])
    assert 200 <= L <= 320
    case = make(workdir, shape, "transit", L)
    default, tile = check_transit(api, case, models_of(case, 600 + L), monkeypatch)
    assert np.array_equal(default, tile)
    # one layer more: refused by transit_init, not by the first batch
    assert layer_limit(api, make(workdir, shape, "transit", L + 1)["cfg"]) == L


def test_eclipse_layer_limit_is_refused_at_init(api, workdir, monkeypatch):
    from oracle import oracle as orc
    # more layers than any eclipse kernel can stage: (nl nf + 96) doubles against 227 KB, nf = 20
    L = layer_limit(api, make(workdir, "tiny", "eclipse", 1500, tempdelt=2600.0)["cfg"])
    assert 1000 < L < 1500
    case = make(workdir, "tiny", "eclipse", L, tempdelt=2600.0)
    models = models_of(case, 700)
    tr = api.Transit(case["cfg"])
    O = orc.Oracle(case["cfg"])
    ref = [O.run(models[m], inter=True) for m in range(models.shape[0])]
    tr.debug_keep(True)
    keep, status = tr.run_batch(models)
    assert (status == 0).all()
    for m, o in enumerate(ref):
        assert np.array_equal(tr.debug_get("last", m).astype(np.int64), o["last"])
        assert relerr(keep[m], o["spectrum"]) < TIGHT
    tr.debug_keep(False)
    # the scan kernel (small batches), the throughput kernel and the slot kernel
    for mode in (None, "0", "1"):
        if mode is None:
            monkeypatch.delenv("BART_ECL_SMALL", raising=False)
        else:
            monkeypatch.setenv("BART_ECL_SMALL", mode)
        spectra, status = tr.run_batch(models)
        assert (status == 0).all()
        for m, o in enumerate(ref):
            assert relerr(spectra[m], o["spectrum"]) < TIGHT, (mode, m)
    monkeypatch.delenv("BART_ECL_SMALL", raising=False)
    tr.free_memory()
    assert layer_limit(api, make(workdir, "tiny", "eclipse", L + 1, tempdelt=2600.0)["cfg"]) == L


# ---- the input converter past one pass (128 layers) and past staging (513 layers, 10 species)
def converter_draws(pt, rng):
    """24 parameter vectors [PT..., log10 CH4 factor] with accepted models and every rejection the
    model can give: temperature bounds, metals past 1 (factor 10^4.2), and -- Madhusudhan-Seager
    -- parameter sets PT.py refuses."""
    if pt == "line":
        p = np.array([-0.5, -0.2, 1.0, 0.0, 1.1]) + rng.normal(0, 0.02, (24, 5))
        p[16:] = rng.uniform([-5.0, -3.0, -2.0, 0.0, 0.55], [2.0, 2.0, 3.0, 1.0, 1.4], (8, 5))
    else:
        # parameter draws of tests/golden/retrieval_pt_smooth.npz (code/PT.py's own verdicts on
        # a grid of the same pressure range)
        g = np.load(os.path.join(cases.GOLDEN_DIR, "retrieval_pt_smooth.npz"))
        key = {"madhu_noinv": "noinv", "madhu_inv": "inv", "piette": "piette"}[pt]
        p = g["%s_pars_a" % key][:24]
    fac = rng.uniform(-2.0, 1.0, (24, 1))
    fac[::7] = 4.2
    return np.hstack([p, fac])


CONVERTER_MODELS = [("line", "const"), ("line", "thorngren"), ("madhu_noinv", "const"),
                    ("madhu_inv", "const"), ("piette", "const")]


@pytest.mark.parametrize("nlayer", [128, 129, 257, 512, 513, 600])
def test_converter_past_one_pass_and_past_staging(nlayer, api, workdir):
    from oracle import retrieval_oracle as ro
    case = make(workdir, "tiny", "eclipse", nlayer)
    tr = api.Transit(case["cfg"])
    rng = np.random.default_rng(nlayer)
    seen = set()
    for pt, tint in CONVERTER_MODELS:
        args = dict(pt_args=cases.W12_PTARGS if pt == "line" else None, tint_type=tint, tmin=400.0,
                    tmax=3000.0)
        tr.converter_init(case["press_bar"], case["species"], case["abund"], ("CH4",), pt, nrad=0, **args)
        conv = ro.Converter(case["press_bar"], case["species"], case["abund"], ("CH4",), pt, **args)
        params = converter_draws(pt, rng)
        prof, status, _ = tr.profiles_from_params(params)
        oprof, ostatus, _ = conv.profiles(params)
        assert np.array_equal(status, ostatus), (pt, tint)
        ok = status == 0
        assert ok.sum() >= 8 and (status == api.REJ_ABUND).any(), (pt, tint)
        assert relerr(prof[ok], oprof[ok]) < 1e-13, (pt, tint)
        seen |= set(status.tolist())
    assert {0, api.REJ_TBOUNDS, api.REJ_ABUND, api.REJ_PTMODEL} <= seen
    if nlayer in (129, 600):
        # parameters -> band fluxes in one call, against converter -> forward model -> band oracle
        wn = tr.get_waveno_arr()
        starwn = np.linspace(wn[0] - 10, wn[-1] + 10, 3000)      # a 6300 K black body
        hc_k = 6.6260755e-27 * 2.99792458e10 / 1.380658e-16
        starfl = 2 * 6.6260755e-27 * 2.99792458e10 ** 2 * starwn ** 3 / np.expm1(hc_k * starwn / 6300.0)
        tr.set_filters(*api.filters_from_files(wn, case["filters"], starwn, starfl), 0.117)
        tr.converter_init(case["press_bar"], case["species"], case["abund"], ("CH4",), "line",
                          pt_args=cases.W12_PTARGS, nrad=0)
        conv = ro.Converter(case["press_bar"], case["species"], case["abund"], ("CH4",), "line",
                            pt_args=cases.W12_PTARGS)
        band = ro.BandOracle(case["cfg"], conv, case["filters"], starwn, starfl, 0.117)
        params = converter_draws("line", rng)
        bf, status = tr.bandflux_from_params(params)
        ref = band(params)
        _, ostatus, _ = conv.profiles(params)
        assert np.array_equal(status, ostatus)
        ok = status == 0
        assert ok.sum() >= 8 and np.all(bf[~ok] == -1.0) and np.all(ref[~ok] == -1.0)
        assert relerr(bf[ok], ref[ok]) < TIGHT
    tr.free_memory()
