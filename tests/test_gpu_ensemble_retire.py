"""GPU: stopping each retrieval of an ensemble at its own convergence.  bart_mcmc_retain
(Transit.mcmc_retain) compacts the device loop to a subset of its retrievals; a kept retrieval must
go on bit for bit as it would have in the larger loop, which is as it would have alone.  The
drivers' grexit="each" stops every retrieval at its own MC3 checkpoint and retains the others.

Lone runs evaluate nchains models per generation and ensembles more; the scan kernel that small
batches take agrees with the other eclipse families to ~1e-10 only, so every comparison pins
BART_ECL_SMALL=0 for both sides."""
import os
import subprocess
import sys

import numpy as np
import pytest

import cases
from test_gpu_retrieval_ensemble import ensemble_inputs, ngpus, same, setup

pytestmark = pytest.mark.gpu
G = cases.GOLDEN_DIR
HERE = os.path.dirname(os.path.abspath(__file__))
NAME = "retr_tiny_eclipse"
STATE = ("params", "currchisq", "numaccept", "outbounds", "bestp", "bestchisq", "bestmodel")
TRACES = ("allparams", "allmodel")


@pytest.fixture(scope="module")
def api(built):
    from bart_b200 import api as a
    a.lib()
    return a


class Loop:
    """An ensemble of retrievals `idx` (of R planned ones) on one Transit, fed host streams (the
    retrievals' own draws) or seeded from keys (700 + r, 1)."""

    def __init__(self, tr, spec, data, uncert, starts, walk, seeded, n, thinning=1, seed=71):
        from bart_b200 import driver
        self.tr, self.walk, self.seeded = tr, walk, seeded
        self.pmin, self.pmax, self.step = (np.array(spec[k], dtype=float) for k in ("pmin", "pmax", "stepsize"))
        self.data, self.uncert, self.starts = data, uncert, np.array(starts)
        free = self.step > 0
        nch, R = spec["nchains"], len(data)
        self.thinning, hsize = thinning, nch + 1
        rng = [np.random.RandomState(seed + r) for r in range(R)]
        if walk == "demc":
            self.draws = [driver.demc_draws(rng[r], nch, n, self.step[free]) for r in range(R)]
        else:
            self.draws = [driver.snooker_draws(rng[r], nch, int(free.sum()), n, hsize, thinning,
                                               self.step[free], self.pmin[free], self.pmax[free])
                          for r in range(R)]
        self.keys = np.array([(700 + r, 1) for r in range(R)], dtype=np.uint64)

    def init(self, idx):
        self.idx, self.lo = list(idx), 0
        self.tr.mcmc_init_ensemble(self.starts[self.idx], self.pmin, self.pmax, self.step,
                                   self.data[self.idx], self.uncert[self.idx], burnin=3)
        if self.seeded:
            self.tr.mcmc_seed(self.keys[self.idx])
        if self.walk == "snooker":
            self.tr.mcmc_snooker_init(np.stack([self.draws[r]["z0"] for r in self.idx]), self.thinning)

    def retain(self, keep):
        self.tr.mcmc_retain(keep)
        self.idx = [self.idx[k] for k in keep]

    def run(self, n):
        from bart_b200 import driver
        lo, hi, sub = self.lo, self.lo + n, [self.draws[r] for r in self.idx]
        if self.seeded:
            self.tr.mcmc_run_seeded(n)
        elif self.walk == "demc":
            self.tr.mcmc_run(*driver.stack_demc_draws(sub, lo, hi))
        else:
            self.tr.mcmc_run_snooker(*driver.stack_snooker_draws(sub, lo, hi))
        self.lo = hi
        return {k: self.tr.mcmc_get(k) for k in TRACES}

    def state(self):
        keys = STATE + (("Z", "Zchisq") if self.walk == "snooker" else ())
        return {k: self.tr.mcmc_get(k) for k in keys}


def equal(a, b, what):
    for k in b:
        assert a[k].shape == b[k].shape and np.array_equal(a[k], b[k], equal_nan=True), (what, k)


def make(api, workdir, R, seed=71):
    case, spec, extra, tr = setup(api, NAME, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % NAME))
    data, uncert, starts, _ = ensemble_inputs(tr, spec, d, R, seed)
    return spec, tr, data, uncert, starts


@pytest.mark.parametrize("walk", ["demc", "snooker"])
@pytest.mark.parametrize("graph", ["1", "0"])
def test_retain_at_once_equals_the_smaller_ensemble(walk, graph, api, workdir, monkeypatch):
    """Init R = 4, retain [1, 3], run: the same as an ensemble initialised with those two."""
    monkeypatch.setenv("BART_MCMC_GRAPH", graph)
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    spec, tr, data, uncert, starts = make(api, workdir, 4)
    n = 12
    L = Loop(tr, spec, data, uncert, starts, walk, False, n)
    L.init(range(4))
    L.retain([1, 3])
    assert api.lib().bart_mcmc_nretr() == 2
    a = L.run(n); a.update(L.state()); a["models"] = tr.mcmc_get("models")
    L.init([1, 3])
    b = L.run(n); b.update(L.state()); b["models"] = tr.mcmc_get("models")
    equal(a, b, walk)
    assert not np.array_equal(a["allparams"][0], a["allparams"][1])
    tr.free_memory()


@pytest.mark.parametrize("seeded", [False, True])
@pytest.mark.parametrize("walk", ["demc", "snooker"])
@pytest.mark.parametrize("graph", ["1", "0"])
def test_retain_sequence_equals_lone_runs(walk, seeded, graph, api, workdir, monkeypatch):
    """n1 generations, retain [0, 2, 3], n2, retain [2] (old retrieval 3), n3: every retrieval's
    traces and state at the moment it leaves equal its lone run's.  Snooker: the history (7 initial
    rows, 122 reserved) outgrows its reservation in the n2 call, after the first retain, so the
    regrown rows come from the compacted template."""
    monkeypatch.setenv("BART_MCMC_GRAPH", graph)
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    spec, tr, data, uncert, starts = make(api, workdir, 4, seed=81)
    n1, n2, n3 = 10, (120 if walk == "snooker" else 14), 9
    L = Loop(tr, spec, data, uncert, starts, walk, seeded, n1 + n2 + n3, seed=81)
    L.init(range(4))
    t1 = L.run(n1)
    L.retain([0, 2, 3])
    t2 = L.run(n2)
    left = L.state()                                   # retrievals 0 and 2 leave here
    L.retain([2])
    with pytest.raises(api.BartError, match="describes the last run call"):
        tr.mcmc_get("allparams")
    t3 = L.run(n3)
    final = L.state()
    assert L.idx == [3]
    for pos, r in enumerate([0, 2, 3]):
        L.init([r])
        lone = [L.run(n1), L.run(n2)]
        if r == 3:
            lone.append(L.run(n3))
            got = {k: np.concatenate([t1[k][3], t2[k][2], t3[k][0]], axis=-1) for k in TRACES}
            st = {k: v[0] for k, v in final.items()}
        else:
            got = {k: np.concatenate([t1[k][r], t2[k][pos]], axis=-1) for k in TRACES}
            st = {k: v[pos] for k, v in left.items()}
        ref = {k: np.concatenate([c[k][0] for c in lone], axis=-1) for k in TRACES}
        equal(got, ref, (r, "traces"))
        equal(st, {k: v[0] for k, v in L.state().items()}, (r, "state"))
    if walk == "snooker":
        assert final["Z"].shape[1] == 7 + n1 + n2 + n3
    assert t1["allparams"].shape[0] == 4 and t2["allparams"].shape[0] == 3
    tr.free_memory()


def test_retain_refusals(api, workdir):
    spec, tr, data, uncert, starts = make(api, workdir, 4)
    n = 6
    L = Loop(tr, spec, data, uncert, starts, "demc", False, 2 * n)
    L.init(range(4))
    for keep, msg in (([], "0 retrievals to keep"), ([0, 1, 2, 3, 3], "5 retrievals to keep"),
                      ([2, 1], "strictly increasing"), ([1, 1], "strictly increasing"),
                      ([0, 4], "not a position"), ([-1], "not a position")):
        with pytest.raises(api.BartError, match=msg):
            tr.mcmc_retain(keep)
    assert api.lib().bart_mcmc_nretr() == 4
    L.retain([0, 1, 2, 3])                              # keeping everything changes nothing
    L.run(n)
    tr.mcmc_get("allparams")
    from bart_b200 import driver
    old = driver.stack_demc_draws(L.draws, n, 2 * n)
    L.retain([0, 2])
    with pytest.raises(api.BartError, match="2 retrievals"):
        tr.mcmc_run(*old)
    for name in ("allparams", "allmodel", "models", "support"):
        with pytest.raises(api.BartError, match="describes the last run call"):
            tr.mcmc_get(name)
    assert tr.mcmc_get("params").shape[0] == 2
    L.run(n)                                            # usable, and fetchable again
    assert tr.mcmc_get("allparams").shape[:2] == (2, spec["nchains"])
    tr.free_memory()
    tr2 = setup(api, NAME, workdir)[3]
    with pytest.raises(api.BartError, match="bart_mcmc_init has not been called"):
        tr2.mcmc_retain([0])
    tr2.free_memory()


def test_retain_returns_the_dropped_history_memory(api, workdir, monkeypatch):
    """Keep 1 of 8 seeded snooker retrievals after 3000 generations: free device memory rises by the
    dropped 7/8 of the history (10.6 MB of Z and Zchisq) to within one 2 MiB granule per history
    array.  The device maps each allocation in 2 MiB granules, and the new arrays (1.3 MB and
    0.2 MB) may land in pages already mapped, so the freed and mapped memory of Z and of Zchisq each
    differ from their exact byte counts by less than one granule: two granules in all."""
    import torch
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    spec, tr, data, uncert, starts = make(api, workdir, 8)
    L = Loop(tr, spec, data, uncert, starts, "snooker", True, 1)      # z0 of the host draws
    L.init(range(8))
    n, nch, npars, hsize = 3000, spec["nchains"], len(spec["params"]), spec["nchains"] + 1
    L.run(n)
    rows = hsize + n + 1                                # snooker_reserve_rows: rows + rows / 2 + 16
    zcap = rows + rows // 2 + 16
    dropped = 7 * zcap * nch * (npars + 1) * 8
    torch.cuda.synchronize()
    before = torch.cuda.mem_get_info()[0]
    L.retain([5])
    after = torch.cuda.mem_get_info()[0]
    granule = 2 << 20
    assert abs((after - before) - dropped) < 2 * granule, (after - before, dropped)
    assert tr.mcmc_get("Z").shape == (1, hsize + n, nch, npars)
    tr.free_memory()


# ---- the drivers: grexit="each" ----
# (start seed, uncertainty scale): the flatter the likelihood the sooner DE-MC's chains mix.  The
# retrieval oracle's DE-MC on these inputs, whose chains are the device's bit for bit, passes MC3's
# test twice in a row at 800, 1000, 1400 and 1200 generations for the flat ones and not at all in
# 2000 for the other two.
PLANTED = ((505, 1e6), (509, 1e6), (500, 1e6), (502, 1e2), (503, 1.0), (504, 1e6), (506, 1e6),
           (507, 1e6), (508, 1e6))
ORACLE_DEMC_LENGTHS = [800, 1000, 1400, 2000, 2000, 1200, 1200, 1200, 1200]


def planted(api, workdir):
    """Golden data with scaled uncertainties; chains start at the truth scattered by 3 step sizes
    drawn from RandomState(seed), whose further draws are the retrieval's streams (`rngs()`)."""
    case, spec, extra, tr = setup(api, NAME, workdir)
    d = np.load(os.path.join(G, "retrieval_mc3_%s.npz" % NAME))
    data = np.repeat(d["data"][None], len(PLANTED), 0)
    uncert = np.array([d["uncert"] * m for _, m in PLANTED])
    pmin, pmax, step = (np.array(spec[k], dtype=float) for k in ("pmin", "pmax", "stepsize"))
    free = step > 0
    truth = np.array(spec["truth"], dtype=float)
    nch = spec["nchains"]

    def rngs():
        gs, starts = [], []
        for seed, _ in PLANTED:
            g = np.random.RandomState(seed)
            p0 = np.repeat(truth[None], nch, 0)
            p0[:, free] += g.normal(0, 3.0, (nch, free.sum())) * step[free]
            gs.append(g)
            starts.append(np.clip(p0, pmin, pmax))
        return gs, starts
    return spec, tr, data, uncert, rngs


@pytest.mark.parametrize("seeded", [False, True])
@pytest.mark.parametrize("walk", ["demc", "snooker"])
def test_grexit_each_equals_lone_grexit_runs(walk, seeded, api, workdir, monkeypatch, tmp_path):
    """Every retrieval of run_<walk>_ensemble(grtest=True, grexit="each") equals run_<walk> of it
    alone with grexit=True, files included; they stop at different checkpoints, some not at all."""
    from bart_b200 import driver
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    spec, tr, data, uncert, rngs = planted(api, workdir)
    R, nch, chainsize, burnin = len(PLANTED), spec["nchains"], 2000, 5
    args = (spec["pmin"], spec["pmax"], spec["stepsize"], chainsize * nch, nch)
    kw = dict(burnin=burnin, grtest=True)
    if walk == "snooker":
        kw["hsize"] = nch + 1
    seeds = [(900 + r, 7) for r in range(R)] if seeded else None
    files = lambda tag: ([str(tmp_path / ("%s%d.npy" % (tag, r))) for r in range(R)],
                         [str(tmp_path / ("%s_model%d.npy" % (tag, r))) for r in range(R)])
    sf, sm = files("ens")
    run = driver.run_demc_ensemble if walk == "demc" else driver.run_snooker_ensemble
    gs, starts = rngs()
    ens = run(tr, data, uncert, starts, *args, rngs=gs, seeds=seeds, savefile=sf, savemodel=sm,
              grexit="each", **kw)
    lone_run = driver.run_demc if walk == "demc" else driver.run_snooker
    lf, lm = files("lone")
    keys = ("allparams", "allmodel", "params", "currchisq", "numaccept", "outbounds", "bestp",
            "bestchisq", "bestmodel", "models", "allstack") + (("Z", "Zchisq") if walk == "snooker" else ())
    lengths = []
    gs, starts = rngs()
    for r in range(R):
        lone = lone_run(tr, data[r], uncert[r], starts[r], *args, rng=gs[r],
                        seed=None if seeds is None else seeds[r], savefile=lf[r], savemodel=lm[r],
                        grexit=True, **kw)
        same(ens[r], lone, keys)
        for a, b in ((sf[r], lf[r]), (sm[r], lm[r])):
            assert np.array_equal(np.load(a), np.load(b))
        lengths.append(lone["allparams"].shape[-1])
    if walk == "demc" and not seeded:
        assert lengths == ORACLE_DEMC_LENGTHS
    early = set(n for n in lengths if n < chainsize)
    assert len(early) >= 2 and chainsize in lengths, lengths
    tr.free_memory()


def test_lone_early_exit_equals_the_shorter_run(api, workdir, monkeypatch):
    """run_demc(grexit=True) that stops at `stop` (800) == run_demc of exactly `stop` generations
    on the first `stop` generations of the same draws."""
    from bart_b200 import driver
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    spec, tr, data, uncert, rngs = planted(api, workdir)
    nch, chainsize = spec["nchains"], 2000
    step = np.array(spec["stepsize"], dtype=float)
    gs, starts = rngs()
    draws = driver.demc_draws(gs[0], nch, chainsize, step[step > 0])
    args = (spec["pmin"], spec["pmax"], step)
    ex = driver.run_demc(tr, data[0], uncert[0], starts[0], *args, chainsize * nch, nch, burnin=5,
                         draws=draws, grtest=True, grexit=True)
    stop = ex["allparams"].shape[-1]
    assert stop == 800
    cut = {k: (v[:stop] if k in ("support", "unif", "ugamma") else v[:, :stop]) for k, v in draws.items()}
    short = driver.run_demc(tr, data[0], uncert[0], starts[0], *args, stop * nch, nch, burnin=5, draws=cut)
    for k in ("allparams", "allmodel", "params", "currchisq", "numaccept", "outbounds", "bestp",
              "bestchisq", "bestmodel", "models", "allstack"):
        assert np.array_equal(np.asarray(ex[k]), np.asarray(short[k])), k
    tr.free_memory()


@pytest.mark.skipif(ngpus() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("p2p", [1, 0])
def test_two_rank_retain_equals_single_gpu(p2p, api, workdir, monkeypatch):
    """R = 4 -> 3 -> 1 over 6 chains moves the rank partition (24 -> 18 -> 6 models): through the
    fused peer window and through NCCL, every rank's output equals the single-GPU run."""
    wd = os.path.join(workdir, "retain_mr_%d" % p2p)
    os.makedirs(wd, exist_ok=True)
    env = dict(os.environ, BART_P2P=str(p2p), BART_ECL_SMALL="0")
    env.pop("LOCAL_RANK", None)
    outs = [os.path.join(wd, "out%d.npz" % r) for r in range(2)]
    procs = [subprocess.Popen([sys.executable, os.path.join(HERE, "retain_rank_worker.py"), str(r), "2", wd,
                               outs[r]], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
             for r in range(2)]
    logs = []
    for p in procs:
        try:
            o, _ = p.communicate(timeout=300)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise AssertionError("retain worker timed out")
        logs.append(o)
    for p, o in zip(procs, logs):
        assert p.returncode == 0, o[-3000:]
    res = [np.load(o) for o in outs]
    monkeypatch.setenv("BART_ECL_SMALL", "0")
    sys.path.insert(0, HERE)
    import retain_rank_worker as w
    single = w.run_sequence(api, os.path.join(wd, "single"), device=0)
    for r in res:
        if p2p:
            assert int(r["p2p"]) == 1, "peer windows were not mapped"
        for k in single:
            assert np.array_equal(r[k], single[k]), k
