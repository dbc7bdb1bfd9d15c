"""TEST INFRASTRUCTURE -- CPU restatement of the random streams of seeded MCMC runs
(bart_mcmc_seed / bart_mcmc_run_seeded; generator and counter layout in bart_b200/csrc/philox.cuh).
Only tests/ import this; the product (bart_b200/) never does.

philox_demc_draws / philox_snooker_draws return the `draws=` dicts oracle/retrieval_oracle.py's
demc() / snooker() take, so a seeded device chain can be reproduced on the CPU.  The Philox core is
pinned against numpy's own np.random.Philox (tests/test_mcmc_device_draws.py).
"""
import numpy as np

# ---- seeded runs: the device's counter-based streams (bart_b200/csrc/philox.cuh) restated ----
# Philox4x64-10 with Random123's constants (numpy's np.random.Philox is an independent
# implementation of the same generator: its random_raw(4) at counter c is the block of c + 1).
_PHILOX_M = (np.uint64(0xD2E7470EE14C6C93), np.uint64(0xCA5A826395121157))
_PHILOX_W = (np.uint64(0x9E3779B97F4A7C15), np.uint64(0xBB67AE8584CAA73B))
_M32 = np.uint64(0xFFFFFFFF)
DRAW_SUPPORT, DRAW_R1, DRAW_R2, DRAW_UNIF, DRAW_UGAMMA = 1, 2, 3, 4, 5
DRAW_I1, DRAW_I2, DRAW_IZ, DRAW_IC, DRAW_USN = 6, 7, 8, 9, 10


def _mulhi64(a, b):
    """High 64 bits of a * b for uint64 arrays (__umul64hi)."""
    s32 = np.uint64(32)
    al, ah, bl, bh = a & _M32, a >> s32, b & _M32, b >> s32
    ll, lh, hl, hh = al * bl, al * bh, ah * bl, ah * bh
    mid = (ll >> s32) + (lh & _M32) + (hl & _M32)
    return hh + (lh >> s32) + (hl >> s32) + (mid >> s32)


def philox4x64_10(ctr, key):
    """Blocks of counters ctr[..., 4] under key (k0, k1): uint64 [..., 4]."""
    c = [np.array(ctr, dtype=np.uint64)[..., j] for j in range(4)]
    k0, k1 = (np.broadcast_to(np.array(k, dtype=np.uint64), c[0].shape).copy() for k in key)
    with np.errstate(over="ignore"):
        for _ in range(10):
            hi0, lo0 = _mulhi64(_PHILOX_M[0], c[0]), _PHILOX_M[0] * c[0]
            hi1, lo1 = _mulhi64(_PHILOX_M[1], c[2]), _PHILOX_M[1] * c[2]
            c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
            k0, k1 = k0 + _PHILOX_W[0], k1 + _PHILOX_W[1]
    return np.stack(c, axis=-1)


def _block(key, purpose, it, chain, element=0, attempt=0):
    """The block of (purpose, global iteration, chain, element, attempt); arguments broadcast."""
    it, chain, element, attempt = np.broadcast_arrays(*(np.asarray(a, dtype=np.int64)
                                                         for a in (it, chain, element, attempt)))
    u = lambda a: a.astype(np.uint64)
    ctr = np.stack([u(element) | (u(attempt) << np.uint64(32)), u(chain), u(it),
                    np.full(it.shape, purpose, np.uint64)], axis=-1)
    return philox4x64_10(ctr, key)


def _u01(x):
    return (x >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def _randint(x, lo, hi):
    return (np.asarray(lo, np.int64) + _mulhi64(x, np.asarray(hi - lo, dtype=np.uint64)).astype(np.int64))


def _normal(key, it, chain, element):
    """numpy's legacy polar method on the (element, attempt) blocks: the device's normals."""
    it, chain, element = np.broadcast_arrays(it, chain, element)
    out = np.full(it.shape, np.nan)
    todo = np.ones(it.shape, bool)
    attempt = 0
    while todo.any():
        b = _block(key, DRAW_SUPPORT, it[todo], chain[todo], element[todo], attempt)
        u, v = 2.0 * _u01(b[..., 0]) - 1.0, 2.0 * _u01(b[..., 1]) - 1.0
        s = u * u + v * v
        ok = (s > 0.0) & (s < 1.0)
        idx = np.flatnonzero(todo)[ok]
        with np.errstate(divide="ignore", invalid="ignore"):
            out.flat[idx] = (u * np.sqrt(-2.0 * np.log(s) / s))[ok]
        todo.flat[idx] = False
        attempt += 1
    return out


def _common_draws(key, nchains, step_free, it_lo, it_hi):
    its = np.arange(it_lo, it_hi)
    nfree = len(step_free)
    it3, c3, f3 = np.meshgrid(its, np.arange(nchains), np.arange(nfree), indexing="ij")
    support = np.asarray(step_free, float) * _normal(key, it3, c3, f3)
    it2, c2 = np.meshgrid(its, np.arange(nchains), indexing="ij")
    unif = _u01(_block(key, DRAW_UNIF, it2, c2)[..., 0])
    ugamma = _u01(_block(key, DRAW_UGAMMA, it2, c2)[..., 0])
    return its, it2, c2, support, unif, ugamma


def philox_demc_draws(key, nchains, step_free, it_lo, it_hi):
    """The streams a seeded DE-MC call draws for global iterations [it_lo, it_hi) under `key`
    (k0, k1), in the shapes demc(draws=...) takes.  MC3's constructions of mcmc.py:498-505: r1 in
    [0, nchains-1) with its own chain swapped for nchains-1, r2 = (c + randint(1, nchains-1)) %
    nchains with r2 == r1 replaced by (c-1) % nchains."""
    if nchains < 3:
        raise ValueError("DE-MC needs at least 3 chains")
    its, it2, c2, support, unif, ugamma = _common_draws(key, nchains, step_free, it_lo, it_hi)
    r1 = _randint(_block(key, DRAW_R1, it2, c2)[..., 0], 0, nchains - 1)
    r1 = np.where(r1 == c2, nchains - 1, r1)
    r2 = (c2 + _randint(_block(key, DRAW_R2, it2, c2)[..., 0], 1, nchains - 1)) % nchains
    r2 = np.where(r2 == r1, (c2 - 1) % nchains, r2)
    return dict(support=support, r1=r1.T.copy(), r2=r2.T.copy(), unif=unif, ugamma=ugamma)


def philox_snooker_draws(key, nchains, nfree, it_lo, it_hi, hsize, thinning, step_free=None):
    """The streams a seeded snooker call draws for global iterations [it_lo, it_hi) of a history
    started at iteration 0 with hsize rows, in the dict snooker(draws=...) takes (without z0, which
    the host draws).  Generation t sees zsize = hsize + ceil(t / thinning) rows; i1, i2 in
    [0, (zsize-1) nchains) with i2 redrawn (next attempt) while it equals i1, iz < zsize-1,
    ic < nchains; the uniform(1.2, 2.2) factors of the chains with ugamma < 0.1 as rows in chain
    order, usn_offset[t - it_lo] their first row.  step_free: the free parameters' step sizes."""
    step_free = np.ones(nfree) if step_free is None else np.asarray(step_free, float)
    its, it2, c2, support, unif, ugamma = _common_draws(key, nchains, step_free, it_lo, it_hi)
    zsize = hsize + (its + thinning - 1) // thinning
    lim = ((zsize - 1) * nchains)[:, None]
    i1 = _randint(_block(key, DRAW_I1, it2, c2)[..., 0], 0, lim)
    i2 = _randint(_block(key, DRAW_I2, it2, c2)[..., 0], 0, lim)
    attempt = 0
    while (i2 == i1).any():
        attempt += 1
        hit = i2 == i1
        i2[hit] = _randint(_block(key, DRAW_I2, it2[hit], c2[hit], 0, attempt)[..., 0], 0, lim.repeat(nchains, 1)[hit])
    iz = _randint(_block(key, DRAW_IZ, it2, c2)[..., 0], 0, (zsize - 1)[:, None])
    ic = _randint(_block(key, DRAW_IC, it2, c2)[..., 0], 0, nchains)
    sj = ugamma < 0.1
    ti, tc = np.nonzero(sj)                                     # row order: generation, then chain
    f = np.arange(nfree)
    usn = 1.2 + (2.2 - 1.2) * _u01(_block(key, DRAW_USN, its[ti][:, None], tc[:, None], f[None, :])[..., 0])
    offset = np.concatenate([[0], np.cumsum(sj.sum(axis=1))]).astype(np.int64)
    return dict(support=support, unif=unif, ugamma=ugamma, i1=i1, i2=i2, iz=iz, ic=ic,
                usnooker=usn.reshape(-1, nfree), usn_offset=offset)
