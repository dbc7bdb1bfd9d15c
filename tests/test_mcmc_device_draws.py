"""CPU: the numpy restatement of the seeded runs' device generator (tests/philox_oracle.py
philox_*; bart_b200/csrc/philox.cuh).  The Philox core is pinned against numpy's own Philox, the
streams against MC3's constraints on them, and their distributions by KS / chi-squared tests."""
import numpy as np
import pytest
from scipy import stats

import philox_oracle as po

KEYS = [(0, 0), (5, 7), (0x0123456789ABCDEF, 0xFEDCBA9876543210), (2 ** 64 - 1, 2 ** 64 - 1)]


@pytest.mark.parametrize("key", KEYS)
def test_philox_core_equals_numpy_philox(key):
    """numpy's random_raw(4) at counter c is the block of c + 1; c0 = 0 exercises the carry of the
    decrement into c1 (numpy counter (2^64-1, c1-1, ...) increments to (0, c1, ...))."""
    ctrs = [(1, 0, 0, 0), (7, 3, 99, 4), (2 ** 40 + 5, 9, 123456, 10), (0, 6, 2, 10),
            (2 ** 64 - 1, 2 ** 64 - 1, 17, 3)]
    for c in ctrs:
        mine = po.philox4x64_10(np.array(c, dtype=np.uint64), key)
        prev = [(c[0] - 1) % 2 ** 64, c[1] if c[0] else c[1] - 1, c[2], c[3]]
        ref = np.random.Philox(key=key[0] + (key[1] << 64),
                               counter=np.array(prev, dtype=np.uint64)).random_raw(4)
        assert np.array_equal(mine, ref), c
    # vectorised counters give the same blocks as one at a time
    many = po.philox4x64_10(np.array(ctrs[:3], dtype=np.uint64), key)
    for j, c in enumerate(ctrs[:3]):
        assert np.array_equal(many[j], po.philox4x64_10(np.array(c, dtype=np.uint64), key))


def test_demc_streams_follow_mc3_constructions():
    for nch in (3, 4, 10, 37):
        d = po.philox_demc_draws((11, nch), nch, np.array([0.1, 2.0, 0.5]), 40, 240)
        n = 200
        assert d["support"].shape == (n, nch, 3) and d["unif"].shape == (n, nch)
        assert d["r1"].shape == (nch, n) and d["r2"].shape == (nch, n)
        c = np.arange(nch)[:, None]
        r1, r2 = d["r1"], d["r2"]
        assert np.all((r1 >= 0) & (r1 < nch) & (r2 >= 0) & (r2 < nch))
        assert np.all(r1 != c) and np.all(r2 != c) and np.all(r2 != r1)
        assert np.all((d["unif"] >= 0) & (d["unif"] < 1) & (d["ugamma"] >= 0) & (d["ugamma"] < 1))
    with pytest.raises(ValueError, match="3 chains"):
        po.philox_demc_draws((1, 2), 2, np.ones(2), 0, 5)


def test_streams_depend_on_iteration_not_on_the_call_split():
    a = po.philox_demc_draws((3, 4), 6, np.ones(2), 0, 50)
    b = po.philox_demc_draws((3, 4), 6, np.ones(2), 20, 50)
    for k in ("support", "unif", "ugamma"):
        assert np.array_equal(a[k][20:], b[k])
    for k in ("r1", "r2"):
        assert np.array_equal(a[k][:, 20:], b[k])
    other = po.philox_demc_draws((3, 5), 6, np.ones(2), 0, 50)
    assert not np.array_equal(a["support"], other["support"])
    s = po.philox_snooker_draws((8, 9), 5, 3, 0, 40, 6, 3)
    t = po.philox_snooker_draws((8, 9), 5, 3, 25, 40, 6, 3)
    for k in ("support", "unif", "ugamma", "i1", "i2", "iz", "ic"):
        assert np.array_equal(s[k][25:], t[k]), k
    o = s["usn_offset"]
    assert np.array_equal(s["usnooker"][o[25]:], t["usnooker"])
    assert np.array_equal(o[25:] - o[25], t["usn_offset"])


@pytest.mark.parametrize("thinning", [1, 3])
def test_snooker_streams_follow_mc3_constructions(thinning):
    nch, nfree, hsize, lo, hi = 10, 7, 11, 5, 605
    d = po.philox_snooker_draws((2026, thinning), nch, nfree, lo, hi, hsize, thinning,
                                np.linspace(0.1, 1, nfree))
    its = np.arange(lo, hi)
    zsize = hsize + np.array([len(range(0, t, thinning)) for t in its])   # rows Z has at iteration t
    lim = (zsize - 1)[:, None]
    assert np.all((d["i1"] >= 0) & (d["i1"] < lim * nch) & (d["i2"] >= 0) & (d["i2"] < lim * nch))
    assert np.all(d["i1"] != d["i2"])
    assert np.all((d["iz"] >= 0) & (d["iz"] < lim)) and np.all((d["ic"] >= 0) & (d["ic"] < nch))
    # the ranges track zsize: late generations reach rows early ones cannot
    assert d["iz"][-50:].max() > lim[0, 0]
    sj = d["ugamma"] < 0.1
    assert np.array_equal(np.diff(d["usn_offset"]), sj.sum(axis=1))
    assert d["usnooker"].shape == (sj.sum(), nfree) and sj.sum() > 0
    assert np.all((d["usnooker"] >= 1.2) & (d["usnooker"] < 2.2))


def test_distributions():
    """About 2e6 draws: support / step is standard normal and the uniforms uniform (KS), r1/r2 pairs
    at MC3's frequencies (chi-squared).  With r1 uniform over the other chains, r2 = (c + k) % n
    with k uniform in [1, n-1) and collisions sent to c-1, the pair (r1, r2) of chain c has the
    probabilities computed here from the construction."""
    nch, nfree = 10, 4
    step = np.array([0.5, 1.0, 2.0, 3.0])
    d = po.philox_demc_draws((777, 1), nch, step, 0, 50000)
    z = (d["support"] / step).ravel()
    assert z.size == 2_000_000
    assert stats.kstest(z, "norm").pvalue > 1e-3
    assert abs(z.mean()) < 3e-3 and abs(z.std() - 1) < 3e-3
    u = np.concatenate([d["unif"].ravel(), d["ugamma"].ravel()])
    assert stats.kstest(u, "uniform").pvalue > 1e-3
    s = po.philox_snooker_draws((777, 2), nch, 2, 0, 2000, 11, 1)
    usn = s["usnooker"].ravel()
    assert stats.kstest((usn - 1.2) / (2.2 - 1.2), "uniform").pvalue > 1e-3
    for c in (0, 4, 9):
        exp = np.zeros((nch, nch))
        for a in range(nch - 1):                  # randint(0, n-1), own chain swapped for n-1
            r1 = nch - 1 if a == c else a
            for k in range(1, nch - 1):
                r2 = (c + k) % nch
                if r2 == r1:
                    r2 = (c - 1) % nch
                exp[r1, r2] += 1.0 / ((nch - 1) * (nch - 2))
        obs = np.zeros((nch, nch))
        np.add.at(obs, (d["r1"][c], d["r2"][c]), 1)
        m = exp > 0
        assert obs[~m].sum() == 0
        assert stats.chisquare(obs[m], exp[m] * obs.sum()).pvalue > 1e-3


def test_driver_refuses_bad_seeds_before_touching_the_device():
    from bart_b200 import driver
    kw = dict(pmin=[0.0], pmax=[1.0], stepsize=[0.1], numit=30, nchains=3)
    data, uncert = np.zeros((2, 4)), np.ones((2, 4))
    with pytest.raises(ValueError, match="mutually exclusive"):
        driver.run_demc_ensemble(None, data, uncert, [[0.5]] * 2, draws=[{}, {}], seeds=[1, 2], **kw)
    with pytest.raises(ValueError, match="mutually exclusive"):
        driver.run_snooker(None, data[0], uncert[0], [0.5], draws={}, seed=1, **kw)
    with pytest.raises(ValueError, match="seeds needs one entry"):
        driver.run_demc_ensemble(None, data, uncert, [[0.5]] * 2, seeds=[1], **kw)
    with pytest.raises(ValueError, match="at least 3 chains"):
        driver.run_demc(None, data[0], uncert[0], [0.5], seed=1, **dict(kw, nchains=2))
    assert driver.seed_key(5) == (5, 0)
    assert driver.seed_key((1 << 64) + 9) == (9, 1)
    assert driver.seed_key(np.array([2 ** 64 - 1, 3], dtype=np.uint64)) == (2 ** 64 - 1, 3)
    for bad in (-1, 1 << 128, (1, 2, 3), (1 << 64, 0)):
        with pytest.raises(ValueError):
            driver.seed_key(bad)


def test_seeded_segments_count_trace_bytes_only():
    from bart_b200 import driver
    R, C, F, D = 64, 10, 9, 40
    cap = driver._segment_cap(R, C, F, D, streams=False)
    assert R * C * cap * 8 * (F + D) <= driver.ENSEMBLE_CALL_BYTES
    assert cap > driver._segment_cap(R, C, F, D)
