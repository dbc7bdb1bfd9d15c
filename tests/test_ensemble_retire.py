"""Host side of grexit="each" (driver.run_segments / _retrieve, no device): a fake Transit serves
planted traces in which retrievals converge at different checkpoints.  Each retrieval must come out
as run_segments(grexit=True) on its own trace, Transit.mcmc_retain must get positions in the
current loop, and the streams of every call must hold the running retrievals only."""
import numpy as np
import pytest

from bart_b200 import driver

R, C, F, P, D, N, BURNIN = 5, 4, 2, 3, 6, 400, 10


def planted_traces():
    """[R][C][F][N]: retrievals 0 and 3 mix from the start, 1 converges late (chains offset in the
    first part), 2 and 4 never converge (chain 0 offset throughout)."""
    rng = np.random.RandomState(12)
    t = rng.normal(size=(R, C, F, N))
    t[1, :, :, :120] += np.arange(C)[:, None, None] * 0.6
    t[2, 0] += 1.0
    t[4, 0] += 1.5
    return t


class FakeTransit:
    """What _retrieve calls on a Transit, for host streams: every array it serves is tagged with
    the original index of the retrieval it belongs to."""

    def __init__(self, traces):
        self.t, self.calls, self.retains, self.live, self.lo = traces, [], [], None, 0

    def mcmc_init_ensemble(self, params, *a, **k):
        self.live = list(range(len(params)))

    def mcmc_run(self, support, r1, r2, unif, ugamma):
        n = unif.shape[1]
        assert unif.shape[0] == len(self.live)
        for k, r in enumerate(self.live):
            assert np.all(unif[k] == r) and np.all(ugamma[k] == r), "streams of the wrong retrieval"
        self.calls.append((self.lo, self.lo + n, list(self.live)))
        self.stale = False
        self.lo += n

    def mcmc_retain(self, keep):
        assert list(keep) == sorted(set(keep)) and 0 <= keep[0] and keep[-1] < len(self.live)
        self.retains.append(list(keep))
        self.live = [self.live[k] for k in keep]
        self.stale = True

    def mcmc_get(self, name):
        if getattr(self, "stale", False) and name in ("allparams", "allmodel", "models"):
            raise AssertionError("%s of the last run call fetched after a retain" % name)
        return self._get(name)

    def _get(self, name):
        lo, hi, live = self.calls[-1]
        assert live == self.live, "fetched after a retain"
        if name == "allparams":
            return self.t[live][..., lo:hi]
        if name == "allmodel":
            return 2 * self.t[live][..., lo:hi]
        shapes = {"params": (C, P), "currchisq": (C,), "numaccept": (C,), "outbounds": (C, F),
                  "bestp": (P,), "bestchisq": (), "bestmodel": (D,), "models": (C, D)}
        return np.array([np.full(shapes[name], float(r)) for r in live])


def tagged_draws():
    return [dict(support=np.zeros((N, C, F)), r1=np.zeros((C, N), int), r2=np.zeros((C, N), int),
                 unif=np.full((N, C), float(r)), ugamma=np.full((N, C), float(r))) for r in range(R)]


def lone_reference(trace):
    """run_segments(grexit=True) on one retrieval's trace, as _retrieve runs a lone retrieval."""
    calls = []
    fetch = lambda: (trace[None][..., calls[-1][0]:calls[-1][1]], 2 * trace[None][..., calls[-1][0]:calls[-1][1]])
    allp, allm, hist, n = driver.run_segments(lambda lo, hi: calls.append((lo, hi)), fetch, N,
                                              burnin=BURNIN, grtest=True, grexit=True)
    return allp[0], allm[0], [(i, p[0]) for i, p in hist], n


def run_each(tr, nretr=R, **kw):
    return driver.run_demc_ensemble(tr, np.zeros((nretr, D)), np.ones((nretr, D)), [np.zeros((C, P))] * nretr,
                                    np.full(P, -9.0), np.full(P, 9.0), np.array([0.1, 0.1, 0.0]), N * C,
                                    C, burnin=BURNIN, draws=tagged_draws()[:nretr], grtest=True,
                                    grexit="each", **kw)


def test_each_retrieval_stops_as_it_would_alone():
    traces = planted_traces()
    tr = FakeTransit(traces)
    outs = run_each(tr)
    lengths = []
    for r, out in enumerate(outs):
        allp, allm, hist, n = lone_reference(traces[r])
        lengths.append(n)
        assert np.array_equal(out["allparams"], allp) and np.array_equal(out["allmodel"], allm)
        assert out["allparams"].shape[-1] == n
        assert len(out["psrf"]) == len(hist)
        for (i, p), (j, q) in zip(out["psrf"], hist):
            assert i == j and np.array_equal(p, q, equal_nan=True)
        assert np.array_equal(out["allstack"], np.hstack([allp[c, :, BURNIN:n] for c in range(C)]))
        for k in ("params", "numaccept", "bestp", "bestmodel", "models", "outbounds", "currchisq"):
            assert np.all(out[k] == r), k          # the state fetched for this retrieval
        assert out["bestchisq"] == float(r)
    # the planted spread: exits at two different checkpoints, and runs to chainsize
    early = sorted(set(n for n in lengths if n < N))
    assert len(early) >= 2 and N in lengths, lengths
    # streams of every call hold the retrievals running then, in order
    for lo, hi, live in tr.calls:
        assert live == [r for r in range(R) if lengths[r] >= hi]
    # retains took positions in the loop as it was then
    live = list(range(R))
    for keep in tr.retains:
        live = [live[k] for k in keep]
    assert live == [r for r in range(R) if lengths[r] == N]
    assert len(tr.retains) == len(early)


@pytest.mark.parametrize("case", ["same_checkpoint", "different_checkpoints", "one_retrieval"])
def test_every_retrieval_stops_early(case):
    """Every retrieval stops before chainsize: at the same checkpoint (identical mixing traces), at
    different ones, or an ensemble of one.  The run ends with the last of them, each equal to its
    lone run_segments(grexit=True); no retain is asked for a loop with nobody left."""
    mixing = np.random.RandomState(3).normal(size=(R, C, F, N))
    traces = {"same_checkpoint": np.repeat(mixing[:1], R, 0), "different_checkpoints": mixing[[0, 3]],
              "one_retrieval": mixing[:1]}[case]
    tr = FakeTransit(traces)
    outs = run_each(tr, len(traces))
    lengths = []
    for r, out in enumerate(outs):
        allp, allm, hist, n = lone_reference(traces[r])
        lengths.append(n)
        assert n < N
        assert np.array_equal(out["allparams"], allp) and np.array_equal(out["allmodel"], allm)
        assert [i for i, _ in out["psrf"]] == [i for i, _ in hist]
        for (i, p), (j, q) in zip(out["psrf"], hist):
            assert np.array_equal(p, q, equal_nan=True)
        assert np.array_equal(out["allstack"], np.hstack([allp[c, :, BURNIN:n] for c in range(C)]))
        assert np.all(out["params"] == r) and out["bestchisq"] == float(r)
    assert tr.calls[-1][1] == max(lengths)
    if case == "different_checkpoints":
        assert len(set(lengths)) == 2 and tr.retains == [[1 if lengths[1] > lengths[0] else 0]]
    else:
        assert len(set(lengths)) == 1 and tr.retains == []


def test_no_retain_after_the_last_checkpoint(monkeypatch):
    """Retrieval 0 passes at the last two checkpoints: it stops with the run, so no retain follows
    (nothing runs after it) and the last call's traces stay fetchable."""
    traces = np.repeat(np.arange(2.0)[:, None, None, None], N, -1) * np.ones((2, C, F, N))
    last = driver.gr_checkpoints(N)[-2]
    monkeypatch.setattr(driver, "gelman_rubin", lambda a: np.full(
        F, 1.0 if a[0, 0, 0] == 0 and a.shape[-1] >= last + 1 - BURNIN else 2.0))
    calls, retired = [], []
    fetch = lambda: (traces[..., calls[-1][0]:calls[-1][1]],) * 2
    out = driver.run_segments(lambda lo, hi: calls.append((lo, hi)), fetch, N, burnin=BURNIN,
                              grtest=True, grexit="each", retire=lambda d, k: retired.append(d))
    assert retired == [] and out[3] == [N, N] and len(out[2][0]) == len(driver.gr_checkpoints(N))


def test_segments_follow_the_smaller_population(monkeypatch):
    """Bounded device calls: after a retain the bound is recomputed for the running retrievals."""
    monkeypatch.setattr(driver, "ENSEMBLE_CALL_BYTES", R * C * 30 * (8 * (2 * F + D + 2) + 8))
    traces = planted_traces()
    tr = FakeTransit(traces)
    outs = run_each(tr)
    for lo, hi, live in tr.calls:
        assert hi - lo <= driver._segment_cap(len(live), C, F, D)
    assert max(hi - lo for lo, hi, live in tr.calls if len(live) < R) > 30
    for r, out in enumerate(outs):
        assert np.array_equal(out["allparams"], lone_reference(traces[r])[0])


def test_grexit_refusals():
    kw = dict(pmin=[0.0], pmax=[1.0], stepsize=[0.1], numit=30, nchains=3)
    for run in (driver.run_demc_ensemble, driver.run_snooker_ensemble):
        with pytest.raises(ValueError, match='grexit="each"'):
            run(None, np.zeros((2, 4)), np.ones((2, 4)), [[0.5]] * 2, grtest=True, grexit=True, **kw)
        with pytest.raises(ValueError, match="needs grtest=True"):
            run(None, np.zeros((2, 4)), np.ones((2, 4)), [[0.5]] * 2, grexit="each", **kw)
    with pytest.raises(ValueError, match="retire"):
        driver.run_segments(lambda lo, hi: None, lambda: None, 10, grtest=True, grexit="each")


def test_legacy_segments_unchanged():
    """Without "each", call boundaries are MC3's checkpoints and multiples of max_segment."""
    calls = []
    trace = np.random.RandomState(1).normal(size=(2, C, F, 95))
    fetch = lambda: (trace[..., calls[-1][0]:calls[-1][1]], trace[..., calls[-1][0]:calls[-1][1]])
    allp, _, hist, n = driver.run_segments(lambda lo, hi: calls.append((lo, hi)), fetch, 95, grtest=True,
                                           max_segment=25)
    cuts = driver.gr_checkpoints(95)
    edges = sorted(set([c + 1 for c in cuts] + [25, 50, 75, 95]))
    assert [hi for _, hi in calls] == edges and n == 95 and np.array_equal(allp, trace)
