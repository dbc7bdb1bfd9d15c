"""GPU: seeded MCMC runs, whose random streams are drawn on the device from per-retrieval Philox
keys (bart_mcmc_seed / bart_mcmc_run_seeded, Transit.mcmc_seed / mcmc_run_seeded, the drivers'
seed= / seeds=).  The device streams equal the numpy restatement (tests/philox_oracle.py), a seeded
run equals the host-stream loop fed its exported streams, and so the oracle's chain; retrieval r of
a seeded ensemble equals the lone run with r's key, however the run is split into calls.

Ensemble-against-lone comparisons pin the eclipse kernel family with BART_ECL_SMALL=0, as
test_gpu_retrieval_ensemble.py does (the lone and ensemble batches differ in size)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import cases
from test_gpu_retrieval_ensemble import (DEMC_KEYS, SNOOKER_KEYS, band_oracle, ensemble_inputs, ngpus,
                                         same, setup)

pytestmark = pytest.mark.gpu
G = cases.GOLDEN_DIR
HERE = os.path.dirname(os.path.abspath(__file__))
KEYS = [(0x243F6A8885A308D3, 0x13198A2E03707344), (7, 0), (2 ** 64 - 1, 12345)]
STREAMS = {"demc": ("support", "unif", "ugamma", "r1", "r2"),
           "snooker": ("support", "unif", "ugamma", "i1", "i2", "iz", "ic", "usnooker", "usn_offset")}


@pytest.fixture(scope="module")
def api(built):
    from bart_b200 import api as a
    a.lib()
    return a


def arrays(spec):
    return tuple(np.array(spec[k], dtype=float) for k in ("pmin", "pmax", "stepsize"))


def init(tr, spec, d, R, walk, seed=55, hsize=None, thinning=1):
    """R retrievals set up on the device (starts / z0 from RandomState(seed + r)); returns the data."""
    from bart_b200 import driver
    pmin, pmax, stepsize = arrays(spec)
    data, uncert, starts, rngs = ensemble_inputs(tr, spec, d, R, seed)
    tr.mcmc_init_ensemble(np.array(starts), pmin, pmax, stepsize, data, uncert, burnin=spec["burnin"])
    if walk == "snooker":
        free = stepsize > 0
        hsize = hsize or spec["nchains"] + 1
        tr.mcmc_snooker_init(np.stack([driver.snooker_z0(rngs[r], spec["nchains"], hsize, pmin[free],
                                                         pmax[free]) for r in range(R)]), thinning)
    return data, uncert, starts


def oracle_streams(walk, key, spec, lo, hi, hsize, thinning):
    import philox_oracle as po
    pmin, pmax, stepsize = arrays(spec)
    step = stepsize[stepsize > 0]
    if walk == "demc":
        return po.philox_demc_draws(key, spec["nchains"], step, lo, hi)
    return po.philox_snooker_draws(key, spec["nchains"], len(step), lo, hi, hsize, thinning, step)


def split_streams(got, walk, R):
    """The ensemble's exported streams -> one dict per retrieval (usnooker sliced, offsets rebased)."""
    out = []
    for r in range(R):
        s = {k: got[k][r] for k in STREAMS[walk] if k != "usnooker"}
        if walk == "snooker":
            o = got["usn_offset"][r]
            s["usnooker"] = got["usnooker"][o[0]:o[-1]]
            s["usn_offset"] = o - o[0]
        out.append(s)
    return out


def assert_streams(dev, ref, walk):
    for k in STREAMS[walk]:
        a, b = np.asarray(dev[k]), np.asarray(ref[k])
        assert a.shape == b.shape, k
        if k == "support":                       # device log: within a few ulp
            assert np.all(np.abs(a - b) <= 4 * np.spacing(np.abs(b))), k
        else:
            assert np.array_equal(a, b), k


@pytest.mark.parametrize("walk", ["demc", "snooker"])
@pytest.mark.parametrize("name", list(cases.RETRIEVAL))
def test_device_streams_equal_oracle(name, walk, api, workdir):
    """R = 1 and 3, two calls each (global iterations 0..n1 and n1..n1+n2): every stream bit for
    bit, support within 4 ulp; snooker with thinning 3 so the index ranges grow across the calls."""
    case, spec, extra, tr = setup(api, name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    hsize, thinning = spec["nchains"] + 1, 3
    for R in (1, 3):
        init(tr, spec, d, R, walk, hsize=hsize, thinning=thinning)
        tr.mcmc_seed(np.array(KEYS[:R], dtype=np.uint64))
        lo = 0
        for n in (7, 12):
            tr.mcmc_run_seeded(n)
            got = {k: tr.mcmc_get(k) for k in STREAMS[walk]}
            assert got["support"].shape == (R, n, spec["nchains"], int((arrays(spec)[2] > 0).sum()))
            assert all(got[k].dtype.kind == "i" for k in STREAMS[walk] if k not in ("support", "unif", "ugamma", "usnooker"))
            for r, s in enumerate(split_streams(got, walk, R)):
                assert_streams(s, oracle_streams(walk, KEYS[r], spec, lo, lo + n, hsize, thinning), walk)
            lo += n
    with pytest.raises(api.BartError, match="snooker run" if walk == "snooker" else "DE-MC run"):
        tr.mcmc_get("r1" if walk == "snooker" else "i1")
    tr.free_memory()


def run_out(tr, walk):
    keys = ("allparams", "allmodel", "params", "numaccept", "outbounds", "bestp", "bestchisq", "currchisq")
    return {k: tr.mcmc_get(k) for k in keys + (("Z", "Zchisq") if walk == "snooker" else ())}


@pytest.mark.parametrize("graph", ["1", "0"])
@pytest.mark.parametrize("walk", ["demc", "snooker"])
@pytest.mark.parametrize("name", list(cases.RETRIEVAL))
def test_seeded_run_replays_through_host_streams(name, walk, graph, api, workdir, monkeypatch):
    """A seeded call equals bart_mcmc_run / bart_mcmc_run_snooker fed the streams it exports:
    traces, allmodel, best fit, Z, acceptance, bit for bit (R = 2, two calls)."""
    from bart_b200 import driver
    monkeypatch.setenv("BART_MCMC_GRAPH", graph)
    case, spec, extra, tr = setup(api, name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    R, calls = 2, (9, 14)
    init(tr, spec, d, R, walk)
    tr.mcmc_seed(np.array(KEYS[:R], dtype=np.uint64))
    seeded, streams = [], []
    for n in calls:
        tr.mcmc_run_seeded(n)
        seeded.append(run_out(tr, walk))
        streams.append({k: tr.mcmc_get(k) for k in STREAMS[walk]})
    init(tr, spec, d, R, walk)
    for n, s, ref in zip(calls, streams, seeded):
        if walk == "demc":
            tr.mcmc_run(s["support"], s["r1"], s["r2"], s["unif"], s["ugamma"])
        else:
            tr.mcmc_run_snooker(s["support"], s["i1"], s["i2"], s["iz"], s["ic"], s["usnooker"],
                                s["usn_offset"], s["unif"], s["ugamma"])
        host = run_out(tr, walk)
        for k in ref:
            assert np.array_equal(host[k], ref[k], equal_nan=True), k
    assert seeded[-1]["numaccept"].sum() > 0
    tr.free_memory()


@pytest.mark.parametrize("walk", ["demc", "snooker"])
@pytest.mark.parametrize("name", list(cases.RETRIEVAL))
def test_seeded_chain_equals_oracle_chain(name, walk, api, workdir):
    """driver.run_demc / run_snooker(seed=k) against the oracle's sampler fed philox_*_draws(k)."""
    from bart_b200 import driver
    from oracle import retrieval_oracle as ro
    case, spec, extra, tr = setup(api, name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    pmin, pmax, stepsize = arrays(spec)
    free = stepsize > 0
    nch, numit = spec["nchains"], spec["numit"]
    chainsize, hsize, thinning, key = int(np.ceil(numit / nch)), nch + 1, 3, KEYS[0]
    starts = driver.start_points(spec["params"], nch, stepsize, pmin, pmax, np.random.RandomState(8))
    args = (pmin, pmax, stepsize, numit, nch)
    band = band_oracle(case, spec, extra)
    if walk == "demc":
        out = driver.run_demc(tr, d["data"], d["uncert"], starts, *args, burnin=spec["burnin"], seed=key)
        ref = ro.demc(band, d["data"], d["uncert"], starts, *args, burnin=spec["burnin"],
                      draws=oracle_streams(walk, key, spec, 0, chainsize, hsize, thinning))
    else:
        out = driver.run_snooker(tr, d["data"], d["uncert"], starts, *args, burnin=spec["burnin"],
                                 thinning=thinning, hsize=hsize, rng=np.random.RandomState(9), seed=key)
        dr = oracle_streams(walk, key, spec, 0, chainsize, hsize, thinning)
        dr["z0"] = driver.snooker_z0(np.random.RandomState(9), nch, hsize, pmin[free], pmax[free])
        ref = ro.snooker(band, d["data"], d["uncert"], starts, *args, burnin=spec["burnin"],
                         thinning=thinning, hsize=hsize, draws=dr)
        assert out["Z"].shape[0] == ref["Zsize"]
        assert np.array_equal(out["Z"], ref["Z"][:ref["Zsize"]])
    for k in ("allparams", "params", "numaccept", "outbounds", "bestp"):
        assert np.array_equal(out[k], ref[k]), k
    assert ref["numaccept"].sum() > 0
    from util import relerr
    assert relerr(out["currchisq"], ref["currchisq"]) < 1e-6
    assert abs(out["bestchisq"] / ref["bestchisq"] - 1) < 1e-6
    tr.free_memory()


@pytest.mark.parametrize("walk", ["demc", "snooker"])
@pytest.mark.parametrize("name", list(cases.RETRIEVAL))
def test_seeded_ensemble_equals_lone_seeded_runs(name, walk, api, workdir, monkeypatch):
    from bart_b200 import driver
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    case, spec, extra, tr = setup(api, name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    R = 3
    data, uncert, starts, _ = ensemble_inputs(tr, spec, d, R, 71, reject_in=1)
    args = (spec["pmin"], spec["pmax"], spec["stepsize"], spec["numit"], spec["nchains"])
    kw = dict(burnin=spec["burnin"])
    if walk == "demc":
        ens = driver.run_demc_ensemble(tr, data, uncert, starts, *args, seeds=KEYS, **kw)
        lone = [driver.run_demc(tr, data[r], uncert[r], starts[r], *args, seed=KEYS[r], **kw) for r in range(R)]
        keys = DEMC_KEYS
    else:
        kw.update(thinning=3)
        rngs = lambda: [np.random.RandomState(500 + r) for r in range(R)]
        ens = driver.run_snooker_ensemble(tr, data, uncert, starts, *args, seeds=KEYS, rngs=rngs(), **kw)
        lone = [driver.run_snooker(tr, data[r], uncert[r], starts[r], *args, seed=KEYS[r], rng=g, **kw)
                for r, g in enumerate(rngs())]
        keys = SNOOKER_KEYS
    for r in range(R):
        same(ens[r], lone[r], keys + ("allstack",))
    assert not np.array_equal(ens[0]["allparams"], ens[1]["allparams"])
    tr.free_memory()


@pytest.mark.parametrize("walk", ["demc", "snooker"])
def test_split_calls_equal_one_call_and_resume_continues_counters(walk, api, workdir, monkeypatch):
    """Calls of 5 + 11 + 8 generations == one call of 24 (traces, state, Z); a resumed DE-MC loop
    (nold = 40) draws the streams of global iterations 40.. ."""
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    name = "retr_tiny_eclipse"
    case, spec, extra, tr = setup(api, name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    R, n = 3, 24
    init(tr, spec, d, R, walk, thinning=2)
    tr.mcmc_seed(np.array(KEYS, dtype=np.uint64))
    tr.mcmc_run_seeded(n)
    one = run_out(tr, walk)
    init(tr, spec, d, R, walk, thinning=2)
    tr.mcmc_seed(np.array(KEYS, dtype=np.uint64))
    parts = []
    for m in (5, 11, 8):
        tr.mcmc_run_seeded(m)
        parts.append(run_out(tr, walk))
    for k in ("allparams", "allmodel"):
        assert np.array_equal(np.concatenate([p[k] for p in parts], axis=-1), one[k]), k
    for k in one:
        if k not in ("allparams", "allmodel"):
            assert np.array_equal(parts[-1][k], one[k], equal_nan=True), k
    if walk == "demc":
        nold = 40
        data, uncert, starts, _ = ensemble_inputs(tr, spec, d, R, 55)
        pmin, pmax, stepsize = arrays(spec)
        tr.mcmc_init_ensemble(one["params"], pmin, pmax, stepsize, data, uncert)
        tr.mcmc_resume(nold, one["allmodel"][..., -1])
        tr.mcmc_seed(np.array(KEYS, dtype=np.uint64))
        tr.mcmc_run_seeded(6)
        got = split_streams({k: tr.mcmc_get(k) for k in STREAMS[walk]}, walk, R)
        for r in range(R):
            assert_streams(got[r], oracle_streams(walk, KEYS[r], spec, nold, nold + 6, 0, 1), walk)
    tr.free_memory()


def test_driver_seeded_snooker_matches_the_stream_path(api, workdir, tmp_path, monkeypatch):
    """run_snooker(seed=) / run_snooker_ensemble(seeds=) return the stream path's keys and write its
    files, and equal the stream path fed the exported streams."""
    from bart_b200 import driver
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    name = "retr_tiny_eclipse"
    case, spec, extra, tr = setup(api, name, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % name))
    pmin, pmax, stepsize = arrays(spec)
    free = stepsize > 0
    nch, numit, hsize = spec["nchains"], spec["numit"], spec["nchains"] + 1
    args = (pmin, pmax, stepsize, numit, nch)
    R = 2
    data, uncert, starts, _ = ensemble_inputs(tr, spec, d, R, 81)
    files = lambda tag: ([str(tmp_path / ("%s%d.npy" % (tag, r))) for r in range(R)],
                         [str(tmp_path / ("%s_model%d.npy" % (tag, r))) for r in range(R)])
    sf, sm = files("seeded")
    lone = driver.run_snooker(tr, data[0], uncert[0], starts[0], *args, hsize=hsize,
                              rng=np.random.RandomState(3), seed=KEYS[0], savefile=sf[0], savemodel=sm[0])
    # the driver's runs are ensembles of one: streams behind [1]
    streams = split_streams({k: tr.mcmc_get(k) for k in STREAMS["snooker"]}, "snooker", 1)[0]
    streams["z0"] = driver.snooker_z0(np.random.RandomState(3), nch, hsize, pmin[free], pmax[free])
    hf, hm = files("host")
    host = driver.run_snooker(tr, data[0], uncert[0], starts[0], *args, hsize=hsize, draws=streams,
                              savefile=hf[0], savemodel=hm[0])
    assert set(lone) == set(host)
    same(lone, host, SNOOKER_KEYS + ("allstack",))
    assert np.array_equal(np.load(sf[0]), np.load(hf[0])) and np.array_equal(np.load(sm[0]), np.load(hm[0]))
    rngs = lambda: [np.random.RandomState(30 + r) for r in range(R)]
    ens = driver.run_snooker_ensemble(tr, data, uncert, starts, *args, hsize=hsize, rngs=rngs(), seeds=KEYS[:R],
                                      savefile=sf, savemodel=sm)
    got = split_streams({k: tr.mcmc_get(k) for k in STREAMS["snooker"]}, "snooker", R)
    for r, g in enumerate(rngs()):
        got[r]["z0"] = driver.snooker_z0(g, nch, hsize, pmin[free], pmax[free])
    hens = driver.run_snooker_ensemble(tr, data, uncert, starts, *args, hsize=hsize, draws=got,
                                       savefile=hf, savemodel=hm)
    for r in range(R):
        assert set(ens[r]) == set(hens[r])
        same(ens[r], hens[r], SNOOKER_KEYS + ("allstack",))
        assert np.array_equal(np.load(sf[r]), np.load(hf[r]))
    # refusals on the device side: no keys, a wrong key count
    tr.mcmc_init_ensemble(np.array(starts), pmin, pmax, stepsize, data, uncert)
    with pytest.raises(api.BartError, match="no keys"):
        tr.mcmc_run_seeded(3)
    with pytest.raises(api.BartError, match="keys must be"):
        tr.mcmc_seed(np.array(KEYS, dtype=np.uint64))
    tr.free_memory()


@pytest.mark.skipif(ngpus() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("p2p", [1, 0])
def test_two_rank_seeded_ensemble_equals_single_gpu(p2p, api, workdir, monkeypatch):
    wd = os.path.join(workdir, "seeded_mr_%d" % p2p)
    os.makedirs(wd, exist_ok=True)
    env = dict(os.environ, BART_P2P=str(p2p), BART_ECL_SMALL="0")
    env.pop("LOCAL_RANK", None)
    worker = os.path.join(HERE, "seeded_ensemble_rank_worker.py")
    outs = [os.path.join(wd, "out%d.npz" % r) for r in range(2)]
    procs = [subprocess.Popen([sys.executable, worker, str(r), "2", wd, outs[r]], env=env,
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    logs = []
    for p in procs:
        try:
            o, _ = p.communicate(timeout=300)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise AssertionError("seeded ensemble worker timed out")
        logs.append(o)
    for p, o in zip(procs, logs):
        assert p.returncode == 0, o[-3000:]
    res = [np.load(o) for o in outs]
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    sys.path.insert(0, HERE)
    import seeded_ensemble_rank_worker as w
    single = w.run_seeded_ensembles(api, os.path.join(wd, "single"), device=0)
    for r in res:
        if p2p:
            assert int(r["p2p"]) == 1, "peer windows were not mapped"
        for k in single:
            assert np.array_equal(r[k], single[k]), k
