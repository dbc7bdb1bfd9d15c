"""GPU: every column-kernel build the launchers can select, against the oracle.

launch_eclipse / launch_transit (kernels.cu) pick a compiled build by configuration: specialised
kernels for 1..4 grid molecules x 0..2 CIA files, the run-time-count build <0, -1> for every other
count, and for eclipse the generic Planck build whenever DevConfig::planck_generic is set.  Eclipse
then picks the scattering / cloud form (SC), the angle form (default ray grid by squaring, or a
run-time angle count) and the kernel: scan, slot, or throughput, whose specialised builds load one
depth ahead up to one resident wave of 8 CTAs per SM and in step above.  Transit picks the
tensor-core or the DFMA tile kernel, each with and without SC.

Each configuration is a small case (40 layers, 2000-2300 cm-1 at step 1, three models) whose grid
molecules and CIA files select one build.  Where the second CIA file (a synthetic H2-He table that
starts at 1000 K) is present, model 1 has a layer at 950 K: the product must reject it with the
oracle's status in every kernel, and the other models' spectra must not depend on it."""
import os

import numpy as np
import pytest

from bart_b200 import synth
from util import relerr, apply_setters

pytestmark = pytest.mark.gpu
TIGHT = 1e-8

# grid molecules by count; the fifth (NH3) joins the atmosphere with 1e-4 taken from H2
MOLS = {1: ["CH4"], 2: ["H2O", "CH4"], 3: ["H2O", "CO", "CH4"], 4: ["H2O", "CO2", "CO", "CH4"],
        5: ["H2O", "CO2", "CO", "CH4", "NH3"]}
SPECIES5 = synth.SPECIES + ["NH3"]
ABUND5 = synth.UNIFORM[:5] + [0.8495] + synth.UNIFORM[6:] + [1e-4]
# (grid molecules, CIA files): every specialised pair, and the run-time-count build reached once by
# the molecule count and once by the CIA-file count
COUNTS = [(n, k) for n in (1, 2, 3, 4) for k in (0, 1, 2)] + [(5, 1), (3, 3)]
ECL_SETTERS = ({}, {"cloudtop": -1.0, "scattering": 1.5})
TR_SETTERS = ({"radius": 94000.0}, {"radius": 94000.0, "cloudtop": -2.0, "scattering": 0.5})
REJECTED = 1                       # the model with a layer below the H2-He table (ncia >= 2)
C2 = 6.6260755e-27 * 2.99792458e10 / 1.380658e-16       # hc/k of column_math.cuh, cm K


def matrix_case(workdir, nmol, ncia, solution="eclipse", raygrid=None, wn=(2000.0, 2300.0)):
    """-> (case, models) of one build configuration (see the module docstring)."""
    tag = "%s_%dmol_%dcia%s_%d" % (solution, nmol, ncia, "_ang" if raygrid else "", int(wn[0]))
    d = os.path.join(workdir, "matrix", tag)
    os.makedirs(d, exist_ok=True)
    kw = dict(shape=dict(wnlow=wn[0], wnhigh=wn[1], wndelt=1.0, mols=MOLS[nmol], toomuch=10.0),
              solution=solution, seed=5000 + 10 * nmol + ncia, nlayer=40, with_cia=ncia > 0,
              cia_h2he=ncia >= 2, extra_cfg=["raygrid %s" % raygrid] if raygrid else None)
    if ncia == 3:              # a second H2-H2 table with its own seed and temperature axis
        t3 = np.array([300.0, 700.0, 1200.0, 1900.0, 2600.0, 3300.0])
        kw["cia_path"] = synth.write_cia(os.path.join(d, "CIA_H2H2_synth.dat")) + "," + \
            synth.write_cia(os.path.join(d, "CIA_H2H2_b.dat"), temps=t3, seed=9)
    if nmol == 5:
        kw.update(species=SPECIES5, abund=ABUND5)
    if solution == "transit":
        kw["refradius_km"] = 95000.0
    case = synth.make_case(d, **kw)
    models = synth.make_models(case, 3, seed=600 + 10 * nmol + ncia, molfit=MOLS[nmol],
                               tmin=1000.0 if ncia >= 2 else 400.0)
    if ncia >= 2:
        models[REJECTED, case["nlayer"] - 1] = 950.0
    return case, models


def oracle_refs(case, models, setters):
    from oracle import oracle as orc
    O = orc.Oracle(case["cfg"])
    apply_setters(O, setters)
    ref = [O.run(m, inter=True) for m in models]
    st = np.array([o["status"] for o in ref], dtype=np.int32)
    return ref, st


def expected_status(ncia, nmodels=3):
    from bart_b200 import api
    st = np.zeros(nmodels, dtype=np.int32)
    if ncia >= 2:
        st[REJECTED] = api.REJ_TCIA
    return st


@pytest.fixture(scope="module")
def api(built):
    from bart_b200 import api as a
    info = a.device_info()
    assert info["cc"][0] >= 10, info
    return a


def check_eclipse(tr, case, models, setters, monkeypatch):
    """Introspection launch, scan, slot and throughput kernels (both forms) against the oracle and
    against each other."""
    ref, st_ref = oracle_refs(case, models, setters)
    ok = st_ref == 0
    okm = np.flatnonzero(ok)
    monkeypatch.delenv("BART_ECL_SMALL", raising=False)
    tr.debug_keep(True)
    keep, st = tr.run_batch(models)
    assert np.array_equal(st, st_ref)
    for m in okm:
        assert np.array_equal(tr.debug_get("last", m).astype(np.int64), ref[m]["last"]), m
        assert relerr(keep[m], ref[m]["spectrum"]) < TIGHT, m
    tr.debug_keep(False)
    out = {}
    for mode in ("2", "1", "0"):
        monkeypatch.setenv("BART_ECL_SMALL", mode)
        out[mode], st = tr.run_batch(models)
        assert np.array_equal(st, st_ref), mode
        assert (out[mode][~ok] == -1.0).all(), mode
        for m in okm:
            assert relerr(out[mode][m], ref[m]["spectrum"]) < TIGHT, (mode, m)
        # the rejected model changes nothing for the others
        alone, st = tr.run_batch(models[ok])
        assert (st == 0).all() and np.array_equal(alone, out[mode][ok]), mode
    assert np.array_equal(out["1"], out["0"])                       # slot == throughput
    assert relerr(out["2"][ok], out["0"][ok]) < 1e-9                # scan: its own approximations
    assert relerr(keep[ok], out["0"][ok]) < 1e-10                   # introspection vs production
    monkeypatch.setenv("BART_ECL_SMALL", "2")
    one, st = tr.run_batch(models[okm[-1]:okm[-1] + 1])
    assert st[0] == 0 and np.array_equal(one[0], out["2"][okm[-1]])
    # a batch past one resident wave of 8 CTAs per SM: the in-step form of the throughput kernel
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    tiles = -(-tr.nwave // 128)
    nbig = 8 * 148 // tiles + 1
    reps = -(-nbig // models.shape[0])
    big, st = tr.run_batch(np.tile(models, (reps, 1))[:nbig])
    assert np.array_equal(st, np.tile(st_ref, reps)[:nbig])
    assert np.array_equal(big, np.tile(out["0"], (reps, 1))[:nbig])
    monkeypatch.delenv("BART_ECL_SMALL")


ECL_PARAMS = [(n, k, None) for n, k in COUNTS] + \
             [(n, k, "0 30 70") for n, k in COUNTS if n in (2, 3) or k in (0, 2)]


@pytest.mark.parametrize("nmol,ncia,raygrid", ECL_PARAMS,
                         ids=["%dmol-%dcia%s" % (n, k, "-3ang" if r else "") for n, k, r in ECL_PARAMS])
def test_eclipse_builds(nmol, ncia, raygrid, api, workdir, monkeypatch):
    case, models = matrix_case(workdir, nmol, ncia, raygrid=raygrid)
    tr = api.Transit(case["cfg"])
    try:
        assert tr.nwave == 301 and tr.nlayer == 40
        for setters in ECL_SETTERS:          # without, then with the scattering / cloud terms
            apply_setters(tr, setters)
            check_eclipse(tr, case, models, setters, monkeypatch)
        _, st_ref = oracle_refs(case, models, {})
        assert np.array_equal(st_ref, expected_status(ncia))
    finally:
        tr.free_memory()


@pytest.mark.parametrize("nmol,ncia", COUNTS, ids=["%dmol-%dcia" % c for c in COUNTS])
def test_transit_builds(nmol, ncia, api, workdir, monkeypatch):
    """Tensor-core and DFMA tile kernels, with and without the scattering / cloud terms."""
    case, models = matrix_case(workdir, nmol, ncia, solution="transit")
    tr = api.Transit(case["cfg"])
    try:
        for setters in TR_SETTERS:
            apply_setters(tr, setters)
            ref, st_ref = oracle_refs(case, models, setters)
            assert np.array_equal(st_ref, expected_status(ncia))
            ok = st_ref == 0
            for mma in (None, "0"):
                if mma is None:
                    monkeypatch.delenv("BART_TRANSIT_MMA", raising=False)
                else:
                    monkeypatch.setenv("BART_TRANSIT_MMA", mma)
                sp, st = tr.run_batch(models)
                assert np.array_equal(st, st_ref), mma
                assert (sp[~ok] == -1.0).all(), mma
                for m in np.flatnonzero(ok):
                    assert relerr(sp[m], ref[m]["spectrum"]) < TIGHT, (mma, m)
            monkeypatch.delenv("BART_TRANSIT_MMA", raising=False)
            tr.debug_keep(True)
            _, st = tr.run_batch(models)
            assert np.array_equal(st, st_ref)
            for m in np.flatnonzero(ok):
                assert np.array_equal(tr.debug_get("last", m).astype(np.int64), ref[m]["last"]), m
            tr.debug_keep(False)
    finally:
        tr.free_memory()


@pytest.mark.parametrize("nmol", [1, 2, 3, 4, 5])
def test_extinction_lookup(nmol, api, workdir):
    """The stand-alone lookup (extinction_kernel<1..4>, and <0> for five molecules)."""
    case, models = matrix_case(workdir, nmol, 1)
    ref, st_ref = oracle_refs(case, models, {})
    assert (st_ref == 0).all()
    tr = api.Transit(case["cfg"])
    try:
        ext = tr.extinction_batch(models, total=False)
        for m in range(models.shape[0]):
            assert relerr(ext[m], ref[m]["ext"]) < 1e-12, m
    finally:
        tr.free_memory()


def wide_planck_case(workdir):
    """2 molecules, 1 CIA file at 120-400 cm-1: hc wn_min / (k T_max) < 0.1 sets planck_generic."""
    case, models = matrix_case(workdir, 2, 1, wn=(120.0, 400.0))
    t = case["grid_temps"]
    x_lo, x_hi = C2 * case["wn"][0] / t[-1], C2 * case["wn"][-1] / t[0]
    assert x_lo < 0.1 or x_hi > 690.0, (x_lo, x_hi)          # transit_init's planck_generic condition
    return case, models


def test_wide_planck_range(api, workdir, monkeypatch):
    case, models = wide_planck_case(workdir)
    tr = api.Transit(case["cfg"])
    try:
        for setters in ECL_SETTERS:
            apply_setters(tr, setters)
            check_eclipse(tr, case, models, setters, monkeypatch)
    finally:
        tr.free_memory()
