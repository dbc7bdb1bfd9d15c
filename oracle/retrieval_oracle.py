"""TEST INFRASTRUCTURE -- CPU restatement of the retrieval loop AROUND the forward model
(SURVEY.md section 8f rows 1 and 2).  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline leg may import this; the product (bart_b200/) never does.

What is restated, in numpy, the literal way:

* input converter  code/BARTfunc.py:309-360  (PT profile, abundance scaling, H2/He
  renormalisation, the temperature-bounds and sum-of-metals rejections, the per-model knobs)
* PT models        code/PT.py:589-739 PT_line + xi (Line et al. 2013 eq. 13-14), PT.py:700-716
  PT_iso, PT.py:741-750 PT_adiabatic, PT.py:157-377 PT_Inversion and 384-586 PT_NoInversion
  (Madhusudhan & Seager 2009), PT.py:752-812 PT_piette
* smoothing        third-party: scipy.ndimage.gaussian_filter1d (scipy 1.18.1 here; kernel
  exp(-x^2 / 2 sigma^2) truncated at int(4 sigma + 0.5) samples and normalised, symmetric
  correlation centre first then outermost pair inwards, edges extended with the end values:
  mode='nearest') and the interpolating degree-1 scipy.interpolate.splrep / splev (FITPACK's
  B-spline basis for k = 1), restated from the published algorithms
* E_2(x)           third-party: scipy.special.expn (scipy 1.18.1 here; cephes `expn.c`, Moshier):
  power series for x <= 1, continued fraction for x > 1, restated from the published algorithm
* chi-squared      modules/MCcubed/src_c/chisq.c:111-142 + include/stats.h:72-103 (priors)
* DE-MC loop       modules/MCcubed/MCcubed/mc/mcmc.py:296-345 (initial state), 484-507 (random
  streams, drawn in MC3's order so a seeded run reproduces MC3's chains), 518-660 (proposal,
  boundary clamp, shared parameters, Metropolis rule, best fit, trace), MPI-mode semantics (every
  chain is evaluated each generation, as BART runs it)

Pinned against the reference itself: tests/golden/retrieval_*.npz are produced by
tests/golden/make_golden_retrieval.py, which imports the reference's code/PT.py and runs the
reference's MCcubed.mc.mcmc (C extensions compiled from a /tmp copy) with fixed seeds.
"""
import numpy as np

EUL = 0.57721566490153286060
MACHEP = 1.11022302462515654042e-16
BIG = 1.44115188075855872e17
MAXLOG = 7.09782712893383996843e2
STEFAN_BOLTZMANN = 5.6703744191844314e-08     # scipy.constants.Stefan_Boltzmann (scipy 1.18)


def expn_scalar(n, x):
    """E_n(x), cephes expn.c algorithm (n small)."""
    if x > MAXLOG:
        return 0.0
    if x == 0.0:
        return np.inf if n < 2 else 1.0 / (n - 1.0)
    if n == 0:
        return np.exp(-x) / x
    if x > 1.0:
        k = 1
        pkm2, qkm2, pkm1, qkm1 = 1.0, x, 1.0, x + n
        ans = pkm1 / qkm1
        while True:
            k += 1
            if k & 1:
                yk, xk = 1.0, n + (k - 1) // 2
            else:
                yk, xk = x, k // 2
            pk = pkm1 * yk + pkm2 * xk
            qk = qkm1 * yk + qkm2 * xk
            if qk != 0:
                r = pk / qk
                t = abs((ans - r) / r)
                ans = r
            else:
                t = 1.0
            pkm2, pkm1, qkm2, qkm1 = pkm1, pk, qkm1, qk
            if abs(pk) > BIG:
                pkm2 /= BIG; pkm1 /= BIG; qkm2 /= BIG; qkm1 /= BIG
            if t <= MACHEP:
                break
        return ans * np.exp(-x)
    psi = -EUL - np.log(x)
    for i in range(1, n):
        psi += 1.0 / i
    z = -x
    xk, yk, pk = 0.0, 1.0, 1.0 - n
    ans = 0.0 if n == 1 else 1.0 / pk
    while True:
        xk += 1.0
        yk *= z / xk
        pk += 1.0
        if pk != 0.0:
            ans += yk / pk
        t = abs(yk / ans) if ans != 0.0 else 1.0
        if t <= MACHEP:
            break
    fact = 1.0
    for i in range(2, n):
        fact *= i
    return z ** (n - 1) * psi / fact - ans


def expn(n, x):
    x = np.asarray(x, dtype=float)
    return np.array([expn_scalar(n, float(v)) for v in x.ravel()]).reshape(x.shape)


def xi(gamma, tau):
    """PT.py:719-737 (eq. 14 of Line et al. 2013)."""
    return (2.0 / 3) * (1 + (1. / gamma) * (1 + (0.5 * gamma * tau - 1) * np.exp(-gamma * tau)) +
                        gamma * (1 - 0.5 * tau ** 2) * expn(2, gamma * tau))


def thorngren_tint(R_star, T_star, sma):
    """PT.py:671-676."""
    T_eq = (R_star / (2.0 * sma)) ** 0.5 * T_star
    F = 4.0 * STEFAN_BOLTZMANN * T_eq ** 4
    return 1.24 * T_eq * np.exp(-(np.log(F) - 0.14) ** 2 / 2.96)


def PT_line(pressure, kappa, gamma1, gamma2, alpha, beta, R_star, T_star, T_int, sma, grav,
            T_int_type="const"):
    """PT.py:589-697."""
    kappa, gamma1, gamma2 = 10 ** kappa, 10 ** gamma1, 10 ** gamma2
    if T_int_type == "thorngren":
        T_int = thorngren_tint(R_star, T_star, sma)
    T_irr = beta * (R_star / (2.0 * sma)) ** 0.5 * T_star
    tau = kappa * (pressure * 1e6) / grav
    xi1, xi2 = xi(gamma1, tau), xi(gamma2, tau)
    return (0.75 * (T_int ** 4 * (2.0 / 3.0 + tau) + T_irr ** 4 * (1 - alpha) * xi1 +
                    T_irr ** 4 * alpha * xi2)) ** 0.25


def PT_iso(p, T):
    return np.ones(len(p)) * T


def PT_adiabatic(p, T0, gamma, logp0):
    p0 = 10 ** logp0
    return T0 / (1 + (gamma - 1) / gamma * np.log(p0 / p))


def gaussian_kernel(sigma):
    """scipy.ndimage._filters._gaussian_kernel1d (order 0) with truncate = 4."""
    radius = int(4.0 * float(sigma) + 0.5)
    x = np.arange(-radius, radius + 1)
    phi = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    return phi / phi.sum()


def gaussian_filter_nearest(v, sigma):
    """gaussian_filter1d(v, sigma, mode='nearest'): NI_Correlate1D's symmetric branch."""
    w = gaussian_kernel(sigma)
    r = len(w) // 2
    n = len(v)
    ext = np.concatenate([np.full(r, v[0]), np.asarray(v, dtype=float), np.full(r, v[-1])])
    out = np.empty(n)
    for l in range(n):
        c = l + r
        t = ext[c] * w[r]
        for j in range(-r, 0):
            t = t + (ext[c + j] + ext[c - j]) * w[r + j]
        out[l] = t
    return out


class NonPhysical(ValueError):
    pass


def PT_NoInversion(p, a1, a2, p1, p3, T3):
    """PT.py:384-586 (p: top -> bottom); raises like the reference when T0, T1 or T3 < 0."""
    p0 = np.amin(p)
    T1 = T3 - (np.log(p3 / p1) / a2) ** 2.0
    T0 = T1 - (np.log(p1 / p0) / a1) ** 2.0
    if T0 < 0 or T1 < 0 or T3 < 0:
        raise NonPhysical()
    T = np.zeros(len(p))
    for i, pi in enumerate(p):
        if p0 <= pi < p1:
            T[i] = (np.log(pi / p0) / a1) ** 2 + T0
        elif p1 <= pi < p3:
            T[i] = (np.log(pi / p1) / a2) ** 2 + T1
        elif p3 <= pi <= np.amax(p):
            T[i] = T3
    return gaussian_filter_nearest(T, 4)


def PT_Inversion(p, a1, a2, p1, p2, p3, T3):
    """PT.py:157-377."""
    p0 = np.amin(p)
    T2 = T3 - (np.log(p3 / p2) / a2) ** 2
    T0 = T2 + (np.log(p1 / p2) / -a2) ** 2 - (np.log(p1 / p0) / a1) ** 2
    T1 = T0 + (np.log(p1 / p0) / a1) ** 2
    if T0 < 0 or T1 < 0 or T2 < 0 or T3 < 0:
        raise NonPhysical()
    T = np.zeros(len(p))
    for i, pi in enumerate(p):
        if p0 <= pi < p1:
            T[i] = (np.log(pi / p0) / a1) ** 2 + T0
        elif p1 <= pi < p2:
            T[i] = (np.log(pi / p2) / -a2) ** 2 + T2
        elif p2 <= pi < p3:
            T[i] = (np.log(pi / p2) / a2) ** 2 + T2
        elif p3 <= pi <= np.amax(p):
            T[i] = T3
    return gaussian_filter_nearest(T, 4)


PIETTE_NODES = (0.01, 0.1, 1.0, 3.2, 10.0, 32.0)


def piette_layers(p):
    """PT.py:787-794: the eight node layers (top, 10 mbar, 0.1, 1, 3.2, 10, 32 bar, bottom)."""
    return np.array([np.argmin(p)] + [np.argmin(np.abs(p - x)) for x in PIETTE_NODES] + [np.argmax(p)])


def PT_piette(p, T0, dTbot_32, dT32_10, dT10_0, dT0_1, dT1_01, dT01_001, dT001_top):
    """PT.py:752-812 (p: top -> bottom, uniform in log p).  Node temperatures, degree-1
    interpolating B-spline in log10 p (splrep k=1 / splev), Gaussian smoothing of 0.3 dex."""
    ilays = piette_layers(p)
    Tn = np.zeros(8)
    Tn[4] = T0
    Tn[5] = T0 + dT10_0
    Tn[6] = Tn[5] + dT32_10
    Tn[7] = Tn[6] + dTbot_32
    Tn[3] = T0 - dT0_1
    Tn[2] = Tn[3] - dT1_01
    Tn[1] = Tn[2] - dT01_001
    Tn[0] = Tn[1] - dT001_top
    x = np.log10(p)
    t = x[ilays]
    if np.any(np.diff(t) <= 0):
        raise ValueError("piette: the pressure grid does not separate the eight node layers")
    T = np.zeros(len(p))
    for i, xi_ in enumerate(x):
        l = min(max(np.searchsorted(t, xi_, side="right") - 1, 0), 6)
        f = 1.0 / (t[l + 1] - t[l])
        T[i] = Tn[l] * (f * (t[l + 1] - xi_)) + Tn[l + 1] * (f * (xi_ - t[l]))
    sig = 0.3 / np.abs(x[0] - x[1])
    return gaussian_filter_nearest(T, sig)


PT_TYPES = {"iso": 0, "line": 1, "adiabatic": 2, "madhu_noinv": 3, "madhu_inv": 4, "piette": 5}
PT_NPARS = {"iso": 1, "line": 5, "adiabatic": 3, "madhu_noinv": 5, "madhu_inv": 6, "piette": 8}
REJ_PTMODEL = 256


class Converter:
    """Input converter of BARTfunc.py:139-222 (set-up) and 320-360 (per proposal)."""

    def __init__(self, pressure_bar, species, abundances, molfit, pt_type, pt_args=None,
                 tint_type="const", tmin=400.0, tmax=3000.0, nrad=0, ncloud=0, nray=0):
        self.press = np.asarray(pressure_bar, dtype=float)          # atmosphere-file order
        self.species = list(species)
        self.base = np.asarray(abundances, dtype=float)             # [layer][species]
        self.nlayer, self.nspec = self.base.shape
        self.imol = [self.species.index(m) for m in molfit]
        self.iH2, self.iHe = self.species.index("H2"), self.species.index("He")
        self.imetals = [i for i, s in enumerate(self.species) if s not in ("H2", "He", "H-", "e-")]
        self.ratio = self.base[:, self.iH2] / self.base[:, self.iHe]
        self.pt_type, self.pt_args, self.tint_type = pt_type, pt_args, tint_type
        self.tmin, self.tmax = tmin, tmax
        self.nrad, self.ncloud, self.nray = nrad, ncloud, nray
        self.npt = PT_NPARS[pt_type]
        # either scattering model takes one slot (polar's value is unused, BARTfunc.py:333-338)
        self.nscat = 1 if nray else 0
        self.npars = self.npt + nrad + ncloud + self.nscat + len(self.imol)

    def temperature(self, ptpars):
        p = self.press[::-1]                                          # BARTfunc.py:176
        if self.pt_type == "line":
            rstar, tstar, tint, sma, grav = self.pt_args
            T = PT_line(p, *ptpars, rstar, tstar, tint, sma, grav, self.tint_type)
        elif self.pt_type == "iso":
            T = PT_iso(p, *ptpars)
        elif self.pt_type == "adiabatic":
            T = PT_adiabatic(p, *ptpars)
        else:
            T = {"madhu_noinv": PT_NoInversion, "madhu_inv": PT_Inversion,
                 "piette": PT_piette}[self.pt_type](p, *ptpars)
        return T[::-1]

    def profiles(self, params):
        """params[M][npars] -> profiles[M][(1+nspec) nlayer], status[M] (0 ok, 16 temperature
        bounds, 32 sum of metals > 1), knobs dict."""
        params = np.atleast_2d(np.asarray(params, dtype=float))
        M = params.shape[0]
        nl, ns = self.nlayer, self.nspec
        prof = np.zeros((M, (ns + 1) * nl))
        status = np.zeros(M, dtype=np.int32)
        off = self.npt + self.nrad + self.ncloud + self.nscat
        for m in range(M):
            try:
                T = self.temperature(params[m, :self.npt])
            except NonPhysical:
                # The reference catches the ValueError and goes on with the profile of the worker's
                # PREVIOUS proposal ("FINDME: what to do here?", BARTfunc.py:323-325); a batch has no
                # previous proposal: the model is rejected (DESIGN.md section 7)
                status[m] = REJ_PTMODEL
                continue
            if np.any(T < self.tmin) or np.any(T > self.tmax) or not np.all(np.isfinite(T)):
                status[m] = 16
                continue
            a = self.base.T.copy()                                    # aprofiles[species][layer]
            for k, i in enumerate(self.imol):
                a[i] = self.base[:, i] * 10.0 ** params[m, off + k]
            q = 1.0 - np.sum(a[self.imetals], axis=0)
            if np.any(q < 0.0):
                status[m] = 32
                continue
            a[self.iH2] = self.ratio * q / (1.0 + self.ratio)
            a[self.iHe] = q / (1.0 + self.ratio)
            prof[m, :nl] = T
            prof[m, nl:] = a.ravel()
        knobs = {}
        c = self.npt
        if self.nrad:
            knobs["refradius"] = params[:, c].copy(); c += 1
        if self.ncloud:
            knobs["cloudtop"] = params[:, c].copy(); c += 1
        if self.nray == 1:
            knobs["scat_flag"] = np.ones(M, dtype=np.int32)
            knobs["scat_logext"] = params[:, c].copy()
        elif self.nray == 2:
            knobs["scat_flag"] = 2 * np.ones(M, dtype=np.int32)
            knobs["scat_logext"] = np.zeros(M)
        return prof, status, knobs


def energy_balance(spectrum, specwn, tstar, rstar, sma, rplanet):
    """code/BARTfunc.py:366-383: -> (e_in, e_out, rejected).  tstar [K]; rstar, sma, rplanet [m]
    (BARTfunc.py:169,369-373); sigma from code/constants.py:19."""
    sig, j2erg = 5.670367e-8, 1e7
    e_in = sig * tstar ** 4 * rstar ** 2 * np.pi * rplanet ** 2 / sma ** 2 * j2erg
    e_out = np.sum(np.diff(specwn) * (spectrum[1:] + spectrum[:-1]) / 2.0) * 4 * (rplanet * 100) ** 2
    return e_in, e_out, bool(e_out > e_in)


def chisq(model, data, uncert, prioroff=None, priorlow=None, priorup=None):
    """chisq.c:111-142 + stats.h:72-103: sequential sums, pow(.,2)."""
    c = 0.0
    for i in range(len(model)):
        c += ((model[i] - data[i]) / uncert[i]) ** 2
    jc = 0.0
    if prioroff is not None:
        for i in range(len(prioroff)):
            if priorlow[i] == -1:
                c += 2.0 * np.log(prioroff[i]); jc += 2.0 * np.log(prioroff[i])
            elif prioroff[i] > 0:
                c += (prioroff[i] / priorup[i]) ** 2
            else:
                c += (prioroff[i] / priorlow[i]) ** 2
    return c, c - jc


def demc(func, data, uncert, params, pmin, pmax, stepsize, numit, nchains, prior=None,
         priorlow=None, priorup=None, burnin=0, fgamma=1.0, fepsilon=0.0, rng=np.random,
         draws=None, resume=None):
    """walk='demc' of mcmc.py, MPI-mode semantics.  resume = (oldparams[nchains][nfree][nold],
    oldmodel[nchains][ndata][nold]): mcmc.py:254-269 -- the chains start from the last state of the
    previous run (no initial jump, no random numbers consumed for it), the traces are appended to the
    old ones, burn-in counts from the old run's first iteration.  `func(params[nchains][npars]) ->
    models[nchains][ndata]`.  Random numbers are drawn from `rng` in MC3's order (mcmc.py:300,
    484-507) unless `draws` supplies them.  Returns a dict with MC3's arrays."""
    data, uncert = np.asarray(data, float), np.asarray(uncert, float)
    params = np.atleast_2d(np.array(params, dtype=float))
    nparams, ndata = params.shape[1], len(data)
    pmin, pmax, stepsize = (np.asarray(a, float) for a in (pmin, pmax, stepsize))
    if prior is None or priorlow is None or priorup is None:
        prior = priorup = priorlow = np.zeros(nparams)
    prior, priorlow, priorup = (np.asarray(a, float) for a in (prior, priorlow, priorup))
    iprior = np.where(priorlow != 0)[0]
    nfree = int(np.sum(stepsize > 0))
    chainsize = int(np.ceil(numit / nchains))
    ifree = np.where(stepsize > 0)[0]
    ishare = np.where(stepsize < 0)[0]
    gamma = fgamma * 2.4 / np.sqrt(2 * nfree)
    nold = 0
    if resume is not None:                                           # mcmc.py:254-267
        oldparams, oldmodel = (np.asarray(a, float) for a in resume)
        nold = oldparams.shape[2]
        params = np.repeat(params, nchains, 0)
        params[:, ifree] = oldparams[:, :, -1]
    if params.shape[0] != nchains:                                   # mcmc.py:296-306
        params = np.repeat(params, nchains, 0)
        for p in ifree:
            params[1:, p] = (draws["init"][p] if draws else
                             rng.normal(params[0, p], stepsize[p], nchains - 1))
            params[np.where(params[:, p] < pmin[p]), p] = pmin[p]
            params[np.where(params[:, p] > pmax[p]), p] = pmax[p]
    for s in ishare:
        params[:, s] = params[:, -int(stepsize[s]) - 1]
    params0 = params.copy()
    models = np.array(func(params), dtype=float).reshape(nchains, ndata)
    currchisq, c2 = np.zeros(nchains), np.zeros(nchains)
    for c in range(nchains):
        currchisq[c], c2[c] = chisq(models[c], data, uncert, (params[c] - prior)[iprior],
                                    priorlow[iprior], priorlow[iprior])
    bestchisq = np.amin(c2)
    bestp = params[np.argmin(c2)].copy()
    bestmodel = models[np.argmin(c2)].copy()
    if draws:
        support, r1, r2, unif, ugamma = (draws[k] for k in ("support", "r1", "r2", "unif", "ugamma"))
    else:                                                            # mcmc.py:484-507
        support = rng.normal(0, stepsize[ifree], (chainsize, nchains, nfree))
        r1 = rng.randint(0, nchains - 1, (nchains, chainsize))
        for c in range(nchains):
            r1[c][np.where(r1[c] == c)] = nchains - 1
        r2 = np.zeros((nchains, chainsize), int)
        for c in range(nchains):
            r2[c] = (c + rng.randint(1, nchains - 1, chainsize)) % nchains
            r2[c][np.where(r2[c] == r1[c])] = (c - 1) % nchains
        unif = rng.uniform(0, 1, (chainsize, nchains))
        ugamma = rng.uniform(0, 1, (chainsize, nchains))
    gamma1 = np.tile(gamma, (nchains, 1))
    nextp = params.copy()
    nextchisq = np.zeros(nchains)
    numaccept = np.zeros(nchains)
    outbounds = np.zeros((nchains, nfree), int)
    allparams = np.zeros((nchains, nfree, chainsize))
    allmodels = np.zeros((chainsize, nchains, ndata))
    allmodel = np.zeros((nchains, ndata, chainsize))          # MC3's savemodel array (mcmc.py:250-252)
    if resume is not None:
        allparams = np.dstack((oldparams, allparams))
        allmodel = np.dstack((oldmodel, allmodel))
    for i in range(chainsize):
        gamma1[ugamma[i] >= 0.1] = gamma
        gamma1[ugamma[i] < 0.1] = 0.98
        jump = gamma1 * (params[r1[:, i]] - params[r2[:, i]])[:, ifree] + fepsilon * support[i]
        nextp[:, ifree] = params[:, ifree] + jump
        outpars = np.asarray(((nextp < pmin) | (nextp > pmax))[:, ifree])
        outflag = np.any(outpars, axis=1)
        outbounds += outpars
        for p in ifree:
            nextp[np.where(nextp[:, p] < pmin[p]), p] = pmin[p]
            nextp[np.where(nextp[:, p] > pmax[p]), p] = pmax[p]
        for s in ishare:
            nextp[:, s] = nextp[:, -int(stepsize[s]) - 1]
        models = np.array(func(nextp), dtype=float).reshape(nchains, ndata)
        allmodels[i] = models
        for c in np.where(~outflag)[0]:
            nextchisq[c], c2[c] = chisq(models[c], data, uncert, (nextp[c] - prior)[iprior],
                                        priorlow[iprior], priorlow[iprior])
        nextchisq[outflag] = np.inf
        with np.errstate(over="ignore", invalid="ignore"):
            accept = np.exp(0.5 * (currchisq - nextchisq))
        accepted = accept >= unif[i]
        if nold + i >= burnin:
            numaccept += accepted
        params[accepted] = nextp[accepted]
        currchisq[accepted] = nextchisq[accepted]
        if np.amin(c2) < bestchisq:
            bestp = params[np.argmin(c2)].copy()
            bestmodel = models[np.argmin(c2)].copy()
            bestchisq = np.amin(c2)
        allparams[:, :, i + nold] = params[:, ifree]
        # mcmc.py:649-651 -- rejected chains keep the previous column; at i = 0 that is column -1,
        # still zeros, so a chain shows zeros until its first accepted proposal (a resumed run
        # continues from the old trace's last column)
        cur = models.copy()
        cur[~accepted] = allmodel[~accepted, :, i + nold - 1]
        allmodel[:, :, i + nold] = cur
    return dict(allparams=allparams, params=params, currchisq=currchisq, numaccept=numaccept,
                outbounds=outbounds, bestp=bestp, bestchisq=bestchisq, bestmodel=bestmodel,
                params0=params0, allmodels=allmodels, allmodel=allmodel,
                draws=dict(support=support, r1=r1, r2=r2, unif=unif, ugamma=ugamma))


def snooker_draws(rng, nchains, nfree, chainsize, hsize, thinning, stepsize_free, pmin_free,
                  pmax_free):
    """The random numbers walk='snooker' consumes, drawn from `rng` in MC3's order: the M0
    initial Z samples (mcmc.py:421-424), support/unif/ugamma (mcmc.py:490-497), then inside
    the loop, per generation, i1, i2 (+ collision redraws), iz, ic (mcmc.py:529-539) and the
    uniform(1.2, 2.2) factors of that generation's snooker chains (mcmc.py:545-556: the two
    calls together take [number of chains with ugamma < 0.1][nfree] values whatever the split
    between projected and unprojected jumps is).  None of it depends on the chain states."""
    z0 = np.zeros((hsize, nchains, nfree))
    for f in range(nfree):
        z0[:, :, f] = rng.uniform(pmin_free[f], pmax_free[f], (hsize, nchains))
    support = rng.normal(0, stepsize_free, (chainsize, nchains, nfree))
    unif = rng.uniform(0, 1, (chainsize, nchains))
    ugamma = rng.uniform(0, 1, (chainsize, nchains))
    sjump = ugamma < 0.1
    i1 = np.zeros((chainsize, nchains), np.int64)
    i2 = np.zeros((chainsize, nchains), np.int64)
    iz = np.zeros((chainsize, nchains), np.int64)
    ic = np.zeros((chainsize, nchains), np.int64)
    usnooker, offset = [], np.zeros(chainsize + 1, np.int64)
    zsize = hsize
    for i in range(chainsize):
        a = rng.randint(0, (zsize - 1) * nchains, nchains)
        b = rng.randint(0, (zsize - 1) * nchains, nchains)
        for j in range(nchains):
            while a[j] == b[j]:
                b[j] = rng.randint(0, (zsize - 1) * nchains)
        i1[i], i2[i] = a, b
        iz[i] = rng.randint(0, zsize - 1, nchains)
        ic[i] = rng.randint(0, nchains, nchains)
        n = int(sjump[i].sum())
        if n:
            usnooker.append(rng.uniform(1.2, 2.2, (n, nfree)))
        offset[i + 1] = offset[i] + n
        if i % thinning == 0:
            zsize += 1
    usn = np.concatenate(usnooker) if usnooker else np.zeros((0, nfree))
    return dict(z0=z0, support=support, unif=unif, ugamma=ugamma, i1=i1, i2=i2, iz=iz, ic=ic,
                usnooker=usn, usn_offset=offset)


def snooker(func, data, uncert, params, pmin, pmax, stepsize, numit, nchains, prior=None,
            priorlow=None, priorup=None, burnin=0, thinning=1, fgamma=1.0, fepsilon=0.0, hsize=1,
            rng=np.random, draws=None):
    """walk='snooker' of mcmc.py (ter Braak & Vrugt 2008 as MC3 implements it), MPI-mode
    semantics (every proposal is evaluated, mcmc.py:582-585), `params` [nchains][npars] given
    per chain.  Random numbers come from `rng` in MC3's order (see snooker_draws) unless
    `draws` supplies them.  Quirks kept: Z rows carry the chains' INITIAL non-free columns
    (mcmc.py:419,425); the Metropolis factor of projected jumps is one Frobenius-norm ratio
    over all such chains of the generation (mcmc.py:606-609)."""
    data, uncert = np.asarray(data, float), np.asarray(uncert, float)
    params = np.atleast_2d(np.array(params, dtype=float))
    nparams, ndata = params.shape[1], len(data)
    pmin, pmax, stepsize = (np.asarray(a, float) for a in (pmin, pmax, stepsize))
    if prior is None or priorlow is None or priorup is None:
        prior = priorup = priorlow = np.zeros(nparams)
    prior, priorlow, priorup = (np.asarray(a, float) for a in (prior, priorlow, priorup))
    iprior = np.where(priorlow != 0)[0]
    nfree = int(np.sum(stepsize > 0))
    chainsize = int(np.ceil(numit / nchains))
    ifree = np.where(stepsize > 0)[0]
    ishare = np.where(stepsize < 0)[0]
    if hsize < nchains:                                              # mcmc.py:233-235
        hsize = nchains + 1
    gamma = fgamma * 2.4 / np.sqrt(2 * nfree)
    if params.shape[0] != nchains:                                   # mcmc.py:296-306
        params = np.repeat(params, nchains, 0)
        for p in ifree:
            params[1:, p] = rng.normal(params[0, p], stepsize[p], nchains - 1)
            params[np.where(params[:, p] < pmin[p]), p] = pmin[p]
            params[np.where(params[:, p] > pmax[p]), p] = pmax[p]
    for s in ishare:
        params[:, s] = params[:, -int(stepsize[s]) - 1]
    params0 = params.copy()
    models = np.array(func(params), dtype=float).reshape(nchains, ndata)
    currchisq, c2 = np.zeros(nchains), np.zeros(nchains)

    def chi(model, p):
        return chisq(model, data, uncert, (p - prior)[iprior], priorlow[iprior], priorlow[iprior])

    for c in range(nchains):
        currchisq[c], c2[c] = chi(models[c], params[c])
    # --- Z set-up, mcmc.py:357-460
    nZchain = int(np.ceil(numit / nchains / thinning))
    Zsize = hsize
    Z = np.zeros((hsize + nZchain, nchains, nparams))
    Zchisq = np.zeros((hsize + nZchain, nchains))
    Z[:, :, :] = params
    if draws is None:
        draws = snooker_draws(rng, nchains, nfree, chainsize, hsize, thinning, stepsize[ifree],
                              pmin[ifree], pmax[ifree])
    for f in range(nfree):
        Z[:hsize, :, ifree[f]] = draws["z0"][:, :, f]
    Z[:, :, stepsize == 0] = params[0, stepsize == 0]
    Zmodels0 = np.zeros((hsize, nchains, ndata))
    for i in range(hsize):
        Zmodels0[i] = np.array(func(Z[i]), dtype=float).reshape(nchains, ndata)
        for c in range(nchains):
            Zchisq[i, c], _ = chi(Zmodels0[i, c], Z[i, c])
    Zibest = np.unravel_index(np.argmin(Zchisq[:hsize]), Zchisq[:hsize].shape)
    bestchisq = np.amin(c2)
    bestp = params[np.argmin(c2)].copy()
    bestmodel = models[np.argmin(c2)].copy()
    if Zchisq[Zibest] < bestchisq:
        bestchisq, bestp, bestmodel = Zchisq[Zibest], Z[Zibest].copy(), Zmodels0[Zibest].copy()
    support, unif, ugamma = draws["support"], draws["unif"], draws["ugamma"]
    sjump = ugamma < 0.1
    nextp = params.copy()
    nextchisq = np.zeros(nchains)
    numaccept = np.zeros(nchains)
    outbounds = np.zeros((nchains, nfree), int)
    allparams = np.zeros((nchains, nfree, chainsize))
    allmodels = np.zeros((chainsize, nchains, ndata))
    allmodel = np.zeros((nchains, ndata, chainsize))          # MC3's savemodel array (mcmc.py:250-252)
    mrfactor = np.zeros(nchains)
    mrtrace = np.ones((chainsize, nchains))
    for i in range(chainsize):
        i1, i2 = draws["i1"][i], draws["i2"][i]
        iz1, ic1 = np.unravel_index(i1, (Zsize, nchains))
        iz2, ic2 = np.unravel_index(i2, (Zsize, nchains))
        z = Z[draws["iz"][i], draws["ic"][i]]
        jump = np.zeros((nchains, nfree))
        noproj = np.all(z == params, axis=1)
        usn = draws["usnooker"][draws["usn_offset"][i]:draws["usn_offset"][i + 1]]
        n_np = int(np.sum(noproj * sjump[i]))
        if n_np != 0:                                                # mcmc.py:544-547
            jump[noproj * sjump[i]] = usn[:n_np] * (Z[iz2, ic2] - Z[iz1, ic1])[noproj * sjump[i]][:, ifree]
        if np.sum(~noproj * sjump[i]) != 0:                          # mcmc.py:549-557
            dz = (params - z)[:, ifree][~noproj * sjump[i]]
            zp1 = np.sum(Z[iz1, ic1][:, ifree][~noproj * sjump[i]] * dz, axis=1)
            zp2 = np.sum(Z[iz2, ic2][:, ifree][~noproj * sjump[i]] * dz, axis=1)
            with np.errstate(divide="ignore", invalid="ignore"):
                jump[~noproj * sjump[i]] = usn[n_np:] * \
                    (zp1 - zp2).reshape(zp1.shape[0], 1) / \
                    np.sum(dz ** 2, axis=1).reshape(zp1.shape[0], 1) * \
                    dz
        jump[~sjump[i]] = gamma * (Z[iz1, ic1] - Z[iz2, ic2])[~sjump[i]][:, ifree] \
            + fepsilon * support[i][~sjump[i]]
        nextp[:, ifree] = params[:, ifree] + jump
        outpars = np.asarray(((nextp < pmin) | (nextp > pmax))[:, ifree])
        outflag = np.any(outpars, axis=1)
        outbounds += outpars
        for p in ifree:
            nextp[np.where(nextp[:, p] < pmin[p]), p] = pmin[p]
            nextp[np.where(nextp[:, p] > pmax[p]), p] = pmax[p]
        for s in ishare:
            nextp[:, s] = nextp[:, -int(stepsize[s]) - 1]
        models = np.array(func(nextp), dtype=float).reshape(nchains, ndata)
        allmodels[i] = models
        for c in np.where(~outflag)[0]:
            nextchisq[c], c2[c] = chi(models[c], nextp[c])
        nextchisq[outflag] = np.inf
        mrfactor[:] = 1.0
        if np.any(sjump[i] * ~noproj * ~outflag):                    # mcmc.py:603-609
            asj = sjump[i] * ~noproj * ~outflag
            mrfactor[asj] = (np.linalg.norm((nextp - z)[:, ifree][asj]) /
                             np.linalg.norm((params - z)[:, ifree][asj])) ** (nfree - 1)
        mrtrace[i] = mrfactor
        with np.errstate(over="ignore", invalid="ignore"):
            accept = np.exp(0.5 * (currchisq - nextchisq)) * mrfactor
        accepted = accept >= unif[i]
        if i >= burnin:
            numaccept += accepted
        params[accepted] = nextp[accepted]
        currchisq[accepted] = nextchisq[accepted]
        if np.amin(c2) < bestchisq:
            bestp = params[np.argmin(c2)].copy()
            bestmodel = models[np.argmin(c2)].copy()
            bestchisq = np.amin(c2)
        allparams[:, :, i] = params[:, ifree]
        cur = models.copy()                                          # mcmc.py:649-651 (see demc)
        cur[~accepted] = allmodel[~accepted, :, i - 1]
        allmodel[:, :, i] = cur
        if i % thinning == 0:                                        # mcmc.py:653-660
            Z[hsize + i // thinning][:, ifree] = params[:, ifree]
            Zchisq[hsize + i // thinning] = currchisq
            Zsize += 1
    return dict(allparams=allparams, params=params, currchisq=currchisq, numaccept=numaccept,
                outbounds=outbounds, bestp=bestp, bestchisq=bestchisq, bestmodel=bestmodel,
                params0=params0, allmodels=allmodels, allmodel=allmodel, Z=Z, Zchisq=Zchisq, Zsize=Zsize,
                hsize=hsize,
                mrfactor=mrtrace, draws=draws)


class BandOracle:
    """params[M][npars] -> band fluxes[M][nfilters]: Converter + forward-model oracle
    (oracle.Oracle, transit_oracle.c) + band integration (oracle.bandflux), i.e. what one
    BARTfunc.py worker returns to MC3 per proposal (BARTfunc.py:309-399), rejected proposals -1."""

    def __init__(self, cfg, converter, filter_files, starwn=None, starfl=None, rprs=1.0):
        from oracle import oracle as orc
        self.orc = orc
        self.O = orc.Oracle(cfg)
        self.conv = converter
        self.wn = self.O.wn
        self.star = starwn is not None
        swn = starwn if self.star else self.wn
        sfl = starfl if self.star else np.ones_like(self.wn)
        self.filters = []
        for f in filter_files:
            fwn, ftr = orc.readfilter(f)
            self.filters.append(orc.resample(self.wn, fwn, ftr, swn, sfl))
        self.rprs = rprs
        self.nfilters = len(self.filters)

    def __call__(self, params):
        params = np.atleast_2d(params)
        prof, status, knobs = self.conv.profiles(params)
        out = -np.ones((params.shape[0], self.nfilters))
        for m in range(params.shape[0]):
            if status[m] or self.O.status(prof[m]):      # rejected: -1 band fluxes, as the product
                continue
            if "refradius" in knobs:
                self.O.set_radius(knobs["refradius"][m])
            if "cloudtop" in knobs:
                self.O.set_cloudtop(knobs["cloudtop"][m])
            if "scat_flag" in knobs:
                self.O.set_scattering(int(knobs["scat_flag"][m]), knobs["scat_logext"][m])
            spec = self.O.run(prof[m])
            out[m] = self.orc.bandflux(spec, self.wn, self.filters, star=self.star, rprs=self.rprs)
        return out
