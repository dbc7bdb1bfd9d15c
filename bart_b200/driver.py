"""Host-side mirror of the MC3 worker / master exchange around the forward model.

* `BandModel` is the per-proposal input and output converter of code/BARTfunc.py:309-399,
  vectorised over a batch of proposals: abundance scaling 10**p with H2/He renormalisation
  (333-347), the temperature-bounds and sum-of-metals rejections (327-330, 339-344: rejected
  proposals return a -1 band-flux vector), per-model radius / cloud-top / scattering knobs
  (350-360), then ONE batched library call profiles -> band fluxes.
* `partition` / `evaluate_generation` replace MC3's one-MPI-process-per-chain Scatter/Gather
  (modules/MCcubed/MCcubed/mc/mcmc.py:583-585, code/BARTfunc.py:312,399): chains are split into
  contiguous blocks, one per rank (= one per GPU); every rank evaluates its block as one batch
  and a single all-gather per generation returns every chain's band fluxes to every rank.
  The communicator is pluggable: a communicator object with `rank`, `world` and `allgather(local, counts)` (the tests bring a
  torch.distributed/gloo one, tests/util.py TorchComm; nccl
  on GPUs) or `LibComm` (the library's own NCCL communicator on device buffers).

`BandModel` takes any callable `pt_func(pressure_bar, pt_params) -> T[layers]` (a caller's own
PT model); for the reference's six PT models (BARTfunc.py:150-155: line, iso, adiabatic, and the
layer-smoothing madhu_noinv, madhu_inv, piette) the whole converter runs on the device: `Transit.converter_init` +
`Transit.bandflux_from_params`, and `run_demc` below keeps MC3's DE-MC generation loop there too.
"""
import numpy as np


def partition(nchains, world, rank):
    """Contiguous block of chains owned by `rank`: sizes differ by at most one."""
    base, extra = divmod(nchains, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


class BandModel:
    def __init__(self, transit, pressure_bar, species, abundances, molfit, pt_func, npt,
                 tmin=400.0, tmax=3000.0, fit_radius=None, fit_cloud=False, fit_scattering=False):
        """abundances[layer, species] in atmosphere-file order (bottom -> top), like
        makeatm.readatm returns; parameters are ordered [PT..., radius?, cloudtop?, scattering?,
        molfit...] as in BARTfunc.py:176-181."""
        self.tr = transit
        self.press = np.asarray(pressure_bar, dtype=float)
        self.species = list(species)
        self.base = np.asarray(abundances, dtype=float)
        self.nlayer, self.nspec = self.base.shape
        self.imol = [self.species.index(m) for m in molfit]
        self.iH2, self.iHe = self.species.index("H2"), self.species.index("He")
        self.imetals = [i for i, s in enumerate(self.species) if s not in ("H2", "He", "H-", "e-")]
        self.ratio = self.base[:, self.iH2] / self.base[:, self.iHe]
        self.pt_func, self.npt = pt_func, npt
        self.tmin, self.tmax = tmin, tmax
        self.nrad = 1 if (fit_radius if fit_radius is not None else not transit.eclipse) else 0
        self.ncloud, self.nray = int(bool(fit_cloud)), int(bool(fit_scattering))

    def profiles(self, params):
        """params[M, npars] -> (profiles[M, (1+nspec)*nlayer], rejected[M] bool, knobs)."""
        params = np.atleast_2d(np.asarray(params, dtype=float))
        M = params.shape[0]
        nl, ns = self.nlayer, self.nspec
        prof = np.zeros((M, (ns + 1) * nl))
        rejected = np.zeros(M, dtype=bool)
        off = self.npt + self.nrad + self.ncloud + self.nray
        for m in range(M):
            T = np.asarray(self.pt_func(self.press[::-1], params[m, :self.npt]))[::-1]
            if np.any(T < self.tmin) or np.any(T > self.tmax) or not np.all(np.isfinite(T)):
                rejected[m] = True
                continue
            q = self.base.copy()
            for k, i in enumerate(self.imol):
                q[:, i] = self.base[:, i] * 10.0 ** params[m, off + k]
            rest = 1.0 - q[:, self.imetals].sum(axis=1)
            if np.any(rest < 0.0):
                rejected[m] = True
                continue
            q[:, self.iH2] = self.ratio * rest / (1.0 + self.ratio)
            q[:, self.iHe] = rest / (1.0 + self.ratio)
            prof[m, :nl] = T
            prof[m, nl:] = q.T.ravel()
        knobs = {}
        c = self.npt
        if self.nrad:
            knobs["refradius"] = params[:, c].copy(); c += 1
        if self.ncloud:
            knobs["cloudtop"] = params[:, c].copy(); c += 1
        if self.nray:
            knobs["scat_flag"] = np.ones(M, dtype=np.int32)
            knobs["scat_logext"] = params[:, c].copy()
        return prof, rejected, knobs

    def evaluate(self, params):
        """Band fluxes [M, nfilters]; rejected proposals get -1 in every band."""
        prof, rejected, knobs = self.profiles(params)
        M = prof.shape[0]
        out = -np.ones((M, self.tr.nfilters))
        ok = np.where(~rejected)[0]
        if len(ok):
            if knobs:
                self.tr.set_batch_knobs(len(ok), **{k: v[ok] for k, v in knobs.items()})
            flux, status = self.tr.bandflux_batch(prof[ok])
            if knobs:
                self.tr.set_batch_knobs(0)
            flux[status != 0] = -1.0
            out[ok] = flux
        return out


class LibComm:
    """All-gather on the library's own NCCL communicator (bart_comm_*), device buffers."""

    def __init__(self, api, rank, world):
        self.api, self.rank, self.world = api, rank, world
        self.cap = 0
        self.d_send = self.d_recv = None

    def allgather(self, local, counts):
        L = self.api.lib()
        width = local.shape[1]
        pad = max(counts)
        n = pad * width
        if n > self.cap:
            for p in (self.d_send, self.d_recv):
                if p:
                    L.bart_dev_free(p)
            self.d_send = L.bart_dev_alloc(n * 8)
            self.d_recv = L.bart_dev_alloc(n * 8 * self.world)
            self.cap = n
        send = np.zeros((pad, width))
        send[:local.shape[0]] = local
        self.api._check(L.bart_memcpy_h2d(self.d_send, send.ctypes.data, n * 8))
        self.api._check(L.bart_comm_allgather(self.d_send, self.d_recv, n))
        recv = np.zeros((self.world, pad, width))
        self.api._check(L.bart_memcpy_d2h(recv.ctypes.data, self.d_recv, n * 8 * self.world))
        return np.concatenate([recv[r, :c] for r, c in enumerate(counts)], axis=0)


# ---------------------------------------------------------------------------------------------
# System parameters of the converter set-up (code/BARTfunc.py:157-172,204-211)
RSUN, RJUP, MJUP = 6.96e8, 7.1492e7, 1.8983e27        # code/constants.py (m, m, kg)
AU, GNEWT = 149597870700.0, 6.6743e-11                # scipy.constants au, G (CODATA 2018)


def read_tep(path):
    """Parameter -> list of value strings of a TEP file (code/reader.py File: `name value uncert
    unit origin  # comment` lines; the first occurrence of a name wins like reader.checkpar)."""
    out = {}
    for line in open(path):
        t = line.split("#", 1)[0].split()
        if t and t[0] not in out:
            out[t[0]] = t[1:]
    return out


def read_atm(atmfile):
    """species, pressure, temperature, abundances[layer][species] of a TEA atmosphere file, with or
    without a radius column -- what code/makeatm.py:753-848 `readatm` hands to BARTfunc.py:185 (the
    converter must see the file's printed pressures and abundances, not the values they were
    rounded from)."""
    lines = open(atmfile).readlines()
    species = lines[lines.index("#SPECIES\n") + 1].split()
    start = lines.index("#TEADATA\n") + 2
    rows = np.array([[float(x) for x in ln.split()] for ln in lines[start:] if ln.strip()])
    first = rows.shape[1] - len(species) - 2               # 1 with a radius column, else 0
    return species, rows[:, first], rows[:, first + 1], rows[:, first + 2:]


def system_from_tep(path, tint=100.0):
    """What BARTfunc.py:157-172 extracts from the TEP file and 204-211 derives from it: stellar
    temperature [K] and radius [m], semi-major axis [m], planetary radius [m] and mass [kg], surface
    gravity [cm s-2]; `pt_args` is the tuple Transit.converter_init takes for PT_line, `rprs` the
    radius ratio of the eclipse band integration (BARTfunc.py:246)."""
    v = read_tep(path)
    tstar = float(v["Ts"][0])
    rstar = float(v["Rs"][0]) * RSUN
    sma = float(v["a"][0]) * AU
    rplanet = float(v["Rp"][0]) * RJUP
    mplanet = float(v["Mp"][0]) * MJUP
    gplanet = 100.0 * GNEWT * mplanet / rplanet ** 2
    return dict(tstar=tstar, rstar=rstar, sma=sma, rplanet=rplanet, mplanet=mplanet, gplanet=gplanet,
                pt_args=(rstar, tstar, float(tint), sma, gplanet), rprs=rplanet / rstar)


class BartWorker:
    """One BART worker (code/BARTfunc.py::main) for a batch of proposals: reads the same `[MCMC]`
    configuration section BARTfunc reads (config_file keys of BARTfunc.py:49-121: tconfig, atmfile,
    PTtype, tint, tint_type, molfit, Tmin, Tmax, filters, tep_name, kurucz, solution, cloudtop,
    scattering, ebalance), sets up transit, the input converter and the output converter on the
    device, and maps parameter vectors [M][npars] to band fluxes [M][nfilters] (rejected proposals:
    -1, like the arrays BARTfunc gathers).  `star=(starwn, starfl)` overrides the Kurucz file."""

    def __init__(self, cfgfile, device=None, star=None, section="MCMC"):
        import configparser
        from . import api
        cp = configparser.ConfigParser(inline_comment_prefixes=("#",))
        cp.optionxform = str
        cp.read([cfgfile])
        get = lambda k, d=None: cp.get(section, k) if cp.has_option(section, k) else d
        self.solution = get("solution")
        if self.solution not in ("transit", "eclipse", "direct"):
            raise ValueError("solution must be transit, eclipse or direct (BARTfunc.py:117)")
        self.molfit = (get("molfit") or "").split()
        pttype = get("PTtype", "none")
        cloudtop, scattering = get("cloudtop"), get("scattering")
        self.tr = tr = api.Transit(get("tconfig"), device=device)
        wn = tr.get_waveno_arr()
        filters = (get("filters") or "").split()
        sysp = system_from_tep(get("tep_name"), tint=float(get("tint", 100.0))) if get("tep_name") else None
        if self.solution in ("eclipse", "transit") and star is None and get("kurucz"):
            logg = float(read_tep(get("tep_name"))["loggstar"][0])
            starfl, starwn, _, _ = api.read_kurucz(get("kurucz"), sysp["tstar"], logg)
            star = (starwn, starfl)
        if self.solution == "eclipse":                       # BARTfunc.py:244-270, 388-391
            tr.set_filters(*api.filters_from_files(wn, filters, star[0], star[1]), sysp["rprs"])
        else:                                                # transit / direct: no stellar division
            start, count, weight, _ = api.filters_from_files(wn, filters)
            tr.set_filters(start, count, weight, None, 1.0)
        species, press, _, abund = read_atm(get("atmfile"))
        nray = 0 if scattering is None else (2 if "polar" in scattering else 1)
        self.npars = tr.converter_init(
            press, species, abund, self.molfit, pttype, pt_args=sysp["pt_args"] if pttype == "line" else None,
            tint_type=get("tint_type", "const"), tmin=float(get("Tmin", 400.0)), tmax=float(get("Tmax", 3000.0)),
            nrad=int(self.solution == "transit"), ncloud=int(cloudtop is not None), nray=nray)
        if str(get("ebalance", "False")).strip() in ("True", "1"):
            tr.set_energy_balance(sysp["tstar"], sysp["rstar"], sysp["sma"], sysp["rplanet"])

    def __call__(self, params):
        return self.tr.bandflux_from_params(params)[0]

    def close(self):
        self.tr.free_memory()


def evaluate_generation(evaluate, params_all, comm):
    """One MCMC generation: `params_all[nchains, npars]` (identical on every rank, as after MC3's
    proposal step) -> band fluxes [nchains, nfilters] on every rank."""
    params_all = np.atleast_2d(params_all)
    nchains = params_all.shape[0]
    lo, hi = partition(nchains, comm.world, comm.rank)
    local = np.asarray(evaluate(params_all[lo:hi]), dtype=float)
    if local.ndim == 1:
        local = local[:, None]
    counts = [partition(nchains, comm.world, r)[1] - partition(nchains, comm.world, r)[0]
              for r in range(comm.world)]
    return comm.allgather(local, counts)


# ---------------------------------------------------------------------------------------------
# MC3's DE-MC sampler around the device-resident generation loop (include/bart_b200.h part 3)
def demc_draws(rng, nchains, chainsize, step_free):
    """The random streams of one run, drawn in MC3's order and shapes
    (modules/MCcubed/MCcubed/mc/mcmc.py:484-507) so that a seeded `rng` (numpy's legacy
    RandomState interface, `numpy.random` itself included) reproduces MC3's chains."""
    nfree = len(step_free)
    support = rng.normal(0, step_free, (chainsize, nchains, nfree))
    r1 = rng.randint(0, nchains - 1, (nchains, chainsize))
    for c in range(nchains):
        r1[c][np.where(r1[c] == c)] = nchains - 1
    r2 = np.zeros((nchains, chainsize), int)
    for c in range(nchains):
        r2[c] = (c + rng.randint(1, nchains - 1, chainsize)) % nchains
        r2[c][np.where(r2[c] == r1[c])] = (c - 1) % nchains
    unif = rng.uniform(0, 1, (chainsize, nchains))
    ugamma = rng.uniform(0, 1, (chainsize, nchains))
    return dict(support=support, r1=r1, r2=r2, unif=unif, ugamma=ugamma)


def start_points(params, nchains, stepsize, pmin, pmax, rng):
    """The chains' starting points (mcmc.py:296-306): `params` as given when it has a row per chain,
    else chain 0 at params[0] and the others scattered around it by normal(0, stepsize) draws from
    `rng`, clipped to [pmin, pmax]."""
    params = np.atleast_2d(np.array(params, dtype=float))
    if params.shape[0] != nchains:
        params = np.repeat(params, nchains, 0)
        for p in np.where(stepsize > 0)[0]:
            params[1:, p] = rng.normal(params[0, p], stepsize[p], nchains - 1)
            params[np.where(params[:, p] < pmin[p]), p] = pmin[p]
            params[np.where(params[:, p] > pmax[p]), p] = pmax[p]
    return params


def run_demc(transit, data, uncert, params, pmin, pmax, stepsize, numit, nchains, prior=None,
             priorlow=None, burnin=0, fgamma=1.0, fepsilon=0.0, rng=np.random, draws=None,
             savefile=None, savemodel=None, grtest=False, grexit=False, thinning=1, resume=False,
             seed=None):
    """`MCcubed.mc.mcmc(..., walk='demc', leastsq=False)` with the whole generation loop on the
    GPU: the host only draws the random streams (once, up front, exactly like mcmc.py does) and
    reads the trace back at the end.  `transit` must have its converter and filters set
    (Transit.converter_init / set_filters).  Returns MC3's arrays: allparams
    [nchains][nfree][chainsize], the stacked posterior after burn-in, bestp, numaccept, ...
    resume=True continues the run whose `savefile` (and `savemodel`) are on disk, like
    mcmc.py:254-269: chains restart from their last states, the new iterations are appended to the
    old traces, burn-in and the convergence test count from the old run's first iteration.
    seed (an int or a pair of uint64 words, see seed_key; not with `draws`): the random streams are
    drawn on the device from that Philox key instead of from `rng` (start points still come from
    `rng`); a resumed seeded run draws from iteration nold on.  The run is an ensemble of one (see
    _retrieve)."""
    old = None
    if resume:
        oldparams = np.load(savefile)
        oldmodel = np.load(savemodel) if savemodel is not None else None
        params = np.repeat(np.atleast_2d(np.array(params, dtype=float))[:1], nchains, 0)
        params[:, np.asarray(stepsize, dtype=float) > 0] = oldparams[:, :, -1]
        allmodel = oldmodel if oldmodel is not None else np.zeros((nchains, len(data), oldparams.shape[2]))
        old = (oldparams[None], allmodel[None], None if oldmodel is None else oldmodel[None, :, :, -1])
    return _retrieve(transit, "demc", np.asarray(data, dtype=float)[None],
                     np.asarray(uncert, dtype=float)[None], [params], pmin, pmax, stepsize, numit,
                     nchains, [rng], None if draws is None else [draws], [savefile], [savemodel],
                     prior=prior, priorlow=priorlow, burnin=burnin, fgamma=fgamma, fepsilon=fepsilon,
                     thinning=thinning, grtest=grtest, grexit=grexit, old=old,
                     seeds=None if seed is None else [seed])[0]


def gelman_rubin(chains):
    """MC3's convergence test (MCcubed/mc/gelman_rubin.py:8-70): potential scale reduction factor of
    every free parameter of chains[nchains][nfree][chainlen]."""
    chains = np.asarray(chains, dtype=float)
    nchains, nfree, chainlen = chains.shape
    W = np.mean(np.var(chains, axis=2), axis=0)
    means = np.mean(chains, axis=2)
    B = (chainlen / (nchains - 1.0)) * np.sum((means - np.mean(means, axis=0)) ** 2, axis=0)
    V = W * ((chainlen - 1.0) / chainlen) + B * ((nchains + 1.0) / (chainlen * nchains))
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.sqrt(V / W)


def gr_checkpoints(chainsize):
    """Iterations i after which MC3 reports / tests convergence: ((i+1) % intsteps == 0) and i > 0
    with intsteps = chainsize / 10 (mcmc.py:238,663; a float in Python 3)."""
    intsteps = chainsize / 10
    return [i for i in range(1, chainsize) if (i + 1) % intsteps == 0]


def run_segments(run, fetch, chainsize, burnin=0, thinning=1, grtest=False, grexit=False, nold=0,
                 old=None, max_segment=None, retire=None):
    """Drive a device-resident walk in the segments MC3's loop is observable in (mcmc.py:662-690).
    `run(lo, hi)` advances generations [lo, hi) (state stays on the device); `fetch()` returns that
    call's allparams / allmodel pieces, [nchains][...][hi - lo] behind any leading axes (the
    driver's traces carry one retrieval axis).  Without grtest it is one segment; `max_segment`
    caps the generations of one call (the host arrays of a call stay bounded).  `old` =
    (allparams, allmodel) of the runs being resumed (nold iterations).  Returns (allparams,
    allmodel, psrf history [(iteration, psrf[leading axes...][nfree])], number of iterations in
    the traces).

    grexit="each" (with grtest, traces [R][nchains][...]): MC3's exit rule for every retrieval on
    its own.  A retrieval whose PSRF passes at two consecutive checkpoints stops there, exactly as
    that retrieval alone with grexit=True would.  `retire(done, keep)` is then called, before the
    next segment, with the positions (in the current fetch) of the retrievals that stop and of those
    that go on (possibly none); it must leave `run` and `fetch` serving the `keep` ones only, and
    returns the `max_segment` of the smaller population (anything when `keep` is empty).  The run ends when every retrieval has stopped or at
    chainsize.  Returns per-retrieval lists, in the original order: (allparams, allmodel, psrf
    history [(iteration, psrf[nfree])], number of iterations in the traces)."""
    each = grexit == "each"
    if each and (not grtest or retire is None):
        raise ValueError('grexit="each" needs grtest=True and a retire callback')
    cuts = gr_checkpoints(chainsize) if grtest else []
    pieces_p, pieces_m, history = [], [], []
    if old is not None:
        pieces_p.append(old[0]); pieces_m.append(old[1])
    live = None                      # "each": original indices of the running retrievals
    lo, grflag = 0, False
    while lo < chainsize:
        hi = min([c + 1 for c in cuts if c + 1 > lo] + [chainsize] +
                 ([(lo // max_segment + 1) * max_segment] if max_segment else []))
        run(lo, hi)
        pp, pm = fetch()
        lo = hi
        i = hi - 1
        if not each:
            pieces_p.append(pp); pieces_m.append(pm)
        else:
            if live is None:         # per retrieval: trace pieces, psrf history, grflag, length
                live = list(range(len(pp)))
                P = [[old[0][r]] if old is not None else [] for r in live]
                M = [[old[1][r]] if old is not None else [] for r in live]
                H, flag, length = [[] for _ in live], [False] * len(live), [nold + chainsize] * len(live)
            for k, r in enumerate(live):
                P[r].append(pp[k]); M[r].append(pm[k])
        if not (grtest and i in cuts and (i + nold) > burnin):
            continue
        if each:
            done = []
            for k, r in enumerate(live):
                psrf = gelman_rubin(np.concatenate(P[r], axis=-1)[..., burnin:i + nold + 1:thinning])
                H[r].append((i, psrf))
                if np.all(psrf < 1.01):
                    if flag[r]:                              # two consecutive passes (mcmc.py:676-683)
                        done.append(k)
                        length[r] = nold + lo
                    flag[r] = True
                else:
                    flag[r] = False
            if done and lo < chainsize:               # at the end nobody needs a smaller loop
                keep = [k for k in range(len(live)) if k not in done]
                max_segment = retire(done, keep)
                live = [live[k] for k in keep]
                if not live:
                    break
            continue
        allp = np.concatenate(pieces_p, axis=-1)[..., burnin:i + nold + 1:thinning]
        lead = allp.shape[:-3]
        psrf = np.array([gelman_rubin(a) for a in allp.reshape((-1,) + allp.shape[-3:])])
        psrf = psrf.reshape(lead + psrf.shape[-1:])
        history.append((i, psrf))
        if np.all(psrf < 1.01):
            if grexit and grflag:                            # two consecutive passes (mcmc.py:676-683)
                break
            grflag = True
        else:
            grflag = False
    if each:
        return ([np.concatenate(p, axis=-1) for p in P], [np.concatenate(m, axis=-1) for m in M], H,
                length)
    return np.concatenate(pieces_p, axis=-1), np.concatenate(pieces_m, axis=-1), history, nold + lo


def _save_mc3_files(out, savefile, savemodel):
    """MC3's output files (mcmc.py:842-850): `savefile` (BART's output.npy, read by
    code/bestFit.py:431 and code/mc3plots.py) = allparams[nchains][nfree][chainsize];
    `savemodel` (BART.cfg: band_eclipse.npy) = allmodel[nchains][ndata][chainsize]."""
    if savefile is not None:
        np.save(savefile, out["allparams"])
    if savemodel is not None:
        np.save(savemodel, out["allmodel"])


def snooker_z0(rng, nchains, hsize, pmin_free, pmax_free):
    """MC3's M0 = hsize x nchains initial history samples (mcmc.py:421-424), uniform in the free
    parameters' bounds, one parameter after the other."""
    z0 = np.zeros((hsize, nchains, len(pmin_free)))
    for f in range(len(pmin_free)):
        z0[:, :, f] = rng.uniform(pmin_free[f], pmax_free[f], (hsize, nchains))
    return z0


def seed_key(seed):
    """The 128-bit Philox key (k0, k1) of a seeded run: an int k in [0, 2^128) is (k mod 2^64,
    k >> 64); a pair of uint64 words is taken as is."""
    if isinstance(seed, (int, np.integer)):
        seed = int(seed)
        if not 0 <= seed < 1 << 128:
            raise ValueError("a seed must be in [0, 2**128)")
        return (seed & 0xFFFFFFFFFFFFFFFF, seed >> 64)
    k = [int(w) for w in seed]
    if len(k) != 2 or not all(0 <= w < 1 << 64 for w in k):
        raise ValueError("a seed is an int or a pair of uint64 words")
    return tuple(k)


def snooker_draws(rng, nchains, nfree, chainsize, hsize, thinning, step_free, pmin_free, pmax_free):
    """The random numbers MC3's walk='snooker' consumes, in its order: the M0 initial history
    samples (mcmc.py:421-424), support / unif / ugamma (490-497), then per generation i1, i2 with
    their collision redraws, iz, ic (529-539) and the uniform(1.2, 2.2) factors of that
    generation's snooker chains (545-556; the reference's two calls take, together,
    [chains with ugamma < 0.1][nfree] values however they split).  None of these depends on the
    chain states, so the host draws them up front and the generation loop stays on the device."""
    z0 = snooker_z0(rng, nchains, hsize, pmin_free, pmax_free)
    support = rng.normal(0, step_free, (chainsize, nchains, nfree))
    unif = rng.uniform(0, 1, (chainsize, nchains))
    ugamma = rng.uniform(0, 1, (chainsize, nchains))
    sjump = ugamma < 0.1
    idx = np.zeros((4, chainsize, nchains), np.int64)
    usn, offset = [], np.zeros(chainsize + 1, np.int64)
    zsize = hsize
    for i in range(chainsize):
        a = rng.randint(0, (zsize - 1) * nchains, nchains)
        b = rng.randint(0, (zsize - 1) * nchains, nchains)
        for j in range(nchains):
            while a[j] == b[j]:
                b[j] = rng.randint(0, (zsize - 1) * nchains)
        idx[0, i], idx[1, i] = a, b
        idx[2, i] = rng.randint(0, zsize - 1, nchains)
        idx[3, i] = rng.randint(0, nchains, nchains)
        n = int(sjump[i].sum())
        if n:
            usn.append(rng.uniform(1.2, 2.2, (n, nfree)))
        offset[i + 1] = offset[i] + n
        if i % thinning == 0:
            zsize += 1
    return dict(z0=z0, support=support, unif=unif, ugamma=ugamma, i1=idx[0], i2=idx[1], iz=idx[2],
                ic=idx[3], usnooker=np.concatenate(usn) if usn else np.zeros((0, nfree)),
                usn_offset=offset)


def run_snooker(transit, data, uncert, params, pmin, pmax, stepsize, numit, nchains, prior=None,
                priorlow=None, burnin=0, thinning=1, fgamma=1.0, fepsilon=0.0, hsize=1,
                rng=np.random, draws=None, savefile=None, savemodel=None, grtest=False, grexit=False,
                seed=None):
    """`MCcubed.mc.mcmc(..., walk='snooker', leastsq=False)` -- the walk BART's examples configure
    -- with the sample history Z, the proposals, the Metropolis rule and the forward models all on
    the GPU.  Returns MC3's arrays (see run_demc) plus Z and Zchisq.  seed: streams drawn on the
    device as in run_demc (start points and the initial history z0 still come from `rng`).  The run
    is an ensemble of one (see _retrieve)."""
    return _retrieve(transit, "snooker", np.asarray(data, dtype=float)[None],
                     np.asarray(uncert, dtype=float)[None], [params], pmin, pmax, stepsize, numit,
                     nchains, [rng], None if draws is None else [draws], [savefile], [savemodel],
                     prior=prior, priorlow=priorlow, burnin=burnin, fgamma=fgamma, fepsilon=fepsilon,
                     thinning=thinning, hsize=hsize, grtest=grtest, grexit=grexit,
                     seeds=None if seed is None else [seed])[0]


# ---------------------------------------------------------------------------------------------
# Every run is an ensemble: R independent retrievals of the same configuration in one device loop
# (Transit.mcmc_init_ensemble), a lone run_demc / run_snooker being R = 1.  Every generation
# evaluates R x nchains models as one batch.  Long runs go through the device in segments of at most
# _segment_cap generations, so the stacked stream and trace arrays of one device call stay under
# ENSEMBLE_CALL_BYTES.  With host streams (the default) total host memory is not bounded: every
# retrieval's streams are drawn up front in MC3's order (what makes its chains MC3's) -- at R = 64,
# 10 chains, 9 free parameters and 1e5 generations the `support` draws alone are 4.6 GB.  Seeded
# runs (seeds=...) draw their streams on the device, call by call, and hold none on the host; in
# either mode the returned traces hold every generation.
ENSEMBLE_CALL_BYTES = 1 << 28          # host stream + trace arrays of one device call


def stack_demc_draws(draws, lo, hi):
    """Transit.mcmc_run's arguments for generations [lo, hi) of R retrievals' demc_draws."""
    h = slice(lo, hi)
    st = lambda k, cols: np.stack([d[k][:, h] if cols else d[k][h] for d in draws])
    return st("support", 0), st("r1", 1), st("r2", 1), st("unif", 0), st("ugamma", 0)


def stack_snooker_draws(draws, lo, hi):
    """Transit.mcmc_run_snooker's arguments for generations [lo, hi) of R retrievals'
    snooker_draws: each retrieval's factor rows one after the other, usn_offset[R][hi-lo+1] rebased
    to absolute rows of the concatenation."""
    h = slice(lo, hi)
    usn, offs, base = [], [], 0
    for d in draws:
        off = np.asarray(d["usn_offset"])[lo:hi + 1]
        usn.append(d["usnooker"][off[0]:off[-1]])
        offs.append(off - off[0] + base)
        base += off[-1] - off[0]
    st = lambda k: np.stack([d[k][h] for d in draws])
    return (st("support"), st("i1"), st("i2"), st("iz"), st("ic"), np.concatenate(usn),
            np.stack(offs), st("unif"), st("ugamma"))


def _segment_cap(nretr, nchains, nfree, ndata, extra=0, streams=True):
    """Generations of one device call so that its host arrays stay under ENSEMBLE_CALL_BYTES
    (streams=False: a seeded call, trace arrays only)."""
    if not streams:
        return max(1, int(ENSEMBLE_CALL_BYTES // (nretr * nchains * 8 * (nfree + ndata))))
    per_gen = nretr * nchains * (8 * (2 * nfree + ndata + 2 + extra) + 2 * 4)
    return max(1, int(ENSEMBLE_CALL_BYTES // per_gen))


def _retrieve(transit, walk, data, uncert, params, pmin, pmax, stepsize, numit, nchains, rngs, draws,
              savefile, savemodel, prior=None, priorlow=None, burnin=0, fgamma=1.0, fepsilon=0.0,
              thinning=1, hsize=1, grtest=False, grexit=False, old=None, seeds=None):
    """R retrievals of `walk` ('demc' or 'snooker') in one device loop.  data / uncert[R][ndata];
    params, rngs, draws, savefile and savemodel one entry per retrieval (rngs, draws, savefile and
    savemodel may also be None); draws that are not given are drawn from the rngs after the start
    points.  `old` = (allparams[R][C][F][nold], allmodel[R][C][D][nold], last model column[R][C][D]
    or None) of the runs being resumed.  seeds: one seed_key argument per retrieval; the streams
    are then drawn on the device from those keys (draws must be None).  Returns R dicts of MC3's
    arrays, each also written to its savefile / savemodel."""
    data = np.asarray(data, dtype=float)
    uncert = np.asarray(uncert, dtype=float)
    nretr = data.shape[0]
    if nretr < 1 or data.ndim != 2 or uncert.shape != data.shape or len(params) != nretr:
        raise ValueError("data, uncert and params need one entry per retrieval")
    for name, v in (("rngs", rngs), ("draws", draws), ("seeds", seeds)):
        if v is not None and len(v) != nretr:
            raise ValueError("%s needs one entry per retrieval (%d)" % (name, nretr))
    if seeds is not None and draws is not None:
        raise ValueError("seed and draws are mutually exclusive: a seeded run draws its streams on "
                         "the device")
    keys = None if seeds is None else np.array([seed_key(s) for s in seeds], dtype=np.uint64)
    if keys is not None and walk == "demc" and nchains < 3:
        raise ValueError("DE-MC needs at least 3 chains (got %d)" % nchains)
    pmin, pmax, stepsize = (np.asarray(a, dtype=float) for a in (pmin, pmax, stepsize))
    ifree = np.where(stepsize > 0)[0]
    chainsize = int(np.ceil(numit / nchains))
    starts = []
    for r in range(nretr):
        rng = rngs[r] if rngs is not None else None
        drawn = draws is None and (keys is None or walk == "snooker")       # streams or z0 from rng
        if rng is None and (np.atleast_2d(params[r]).shape[0] != nchains or drawn):
            raise ValueError("retrieval %d needs an rng (its start points or random streams are "
                             "drawn)" % r)
        starts.append(start_points(params[r], nchains, stepsize, pmin, pmax, rng))
    transit.mcmc_init_ensemble(np.array(starts), pmin, pmax, stepsize, data, uncert, prior=prior,
                               priorlow=priorlow, fgamma=fgamma, fepsilon=fepsilon, burnin=burnin)
    nold = 0 if old is None else old[0].shape[-1]
    if old is not None:
        transit.mcmc_resume(nold, old[2])
    if keys is not None:
        transit.mcmc_seed(keys)
    active = list(range(nretr))          # the loop's retrievals (grexit="each" retains a subset)
    if walk == "demc":
        if keys is not None:
            run = lambda lo, hi: transit.mcmc_run_seeded(hi - lo)
        else:
            if draws is None:
                draws = [demc_draws(rng, nchains, chainsize, stepsize[ifree]) for rng in rngs]
            run = lambda lo, hi: transit.mcmc_run(*stack_demc_draws([draws[r] for r in active], lo, hi))
        zkeys, extra = (), 0
    else:
        if hsize < nchains:                                          # mcmc.py:233-235
            hsize = nchains + 1
        if keys is not None:
            z0 = np.stack([snooker_z0(rng, nchains, hsize, pmin[ifree], pmax[ifree]) for rng in rngs])
            run = lambda lo, hi: transit.mcmc_run_seeded(hi - lo)
        else:
            if draws is None:
                draws = [snooker_draws(rng, nchains, len(ifree), chainsize, hsize, thinning,
                                       stepsize[ifree], pmin[ifree], pmax[ifree]) for rng in rngs]
            z0 = np.stack([d["z0"] for d in draws])
            run = lambda lo, hi: transit.mcmc_run_snooker(
                *stack_snooker_draws([draws[r] for r in active], lo, hi))
        transit.mcmc_snooker_init(z0, thinning)
        zkeys, extra = ("Z", "Zchisq"), len(ifree) / 5 + 2
    cap = lambda n: _segment_cap(n, nchains, len(ifree), data.shape[1], extra, streams=keys is None)
    state = {}                            # original index -> final state of the loop's arrays

    def take_state(positions):
        got = {k: transit.mcmc_get(k) for k in ("params", "currchisq", "numaccept", "outbounds", "bestp",
                                                "bestchisq", "bestmodel", "models") + zkeys}
        for k in positions:
            state[active[k]] = {name: v[k] for name, v in got.items()}

    def retire(done, keep):               # grexit="each": `done` stop, the loop keeps `keep`
        take_state(done)
        if keep:
            transit.mcmc_retain(keep)
        active[:] = [active[k] for k in keep]
        return cap(len(active)) if active else None     # none left: the run ends here

    allp, allm, history, chainlen = run_segments(
        run, lambda: (transit.mcmc_get("allparams"), transit.mcmc_get("allmodel")), chainsize,
        burnin=burnin, thinning=thinning, grtest=grtest, grexit=grexit, nold=nold,
        old=None if old is None else old[:2], max_segment=cap(nretr), retire=retire)
    if active:
        take_state(range(len(active)))
    if grexit != "each":                  # one length and psrf history for all: split them
        history = [[(i, psrf[r]) for i, psrf in history] for r in range(nretr)]
        chainlen = [chainlen] * nretr
    outs = []
    for r in range(nretr):
        out = dict(state[r])
        out["allparams"], out["allmodel"] = allp[r], allm[r]
        out["psrf"] = history[r]
        out["bestchisq"] = float(out.pop("bestchisq"))
        out["allstack"] = np.hstack([allp[r][c, :, burnin:chainlen[r]] for c in range(nchains)])  # mcmc.py:692-695
        _save_mc3_files(out, savefile[r] if savefile is not None else None,
                        savemodel[r] if savemodel is not None else None)
        outs.append(out)
    return outs


def run_demc_ensemble(transit, data, uncert, params, pmin, pmax, stepsize, numit, nchains,
                      prior=None, priorlow=None, burnin=0, fgamma=1.0, fepsilon=0.0, rngs=None,
                      draws=None, savefile=None, savemodel=None, grtest=False, grexit=False,
                      thinning=1, seeds=None):
    """`run_demc` for R retrievals of the same configuration in one device loop: data /
    uncert[R][ndata], params[R] (each what run_demc takes: one start point, scattered with that
    retrieval's rng as mcmc.py:296-306 does, or one row per chain), rngs / draws one per retrieval
    (draws as demc_draws returns them), savefile / savemodel one path per retrieval.  Returns a list
    of R dicts with run_demc's keys; retrieval r equals run_demc on its own data and streams.
    seeds: one seed per retrieval (see run_demc's seed; not with draws); retrieval r then equals
    run_demc with seed=seeds[r].
    grexit="each" (with grtest=True) stops every retrieval at its own convergence, by MC3's rule
    (two consecutive checkpoints with every PSRF < 1.01): its outputs are then those of run_demc
    with grexit=True on its own, and the retrievals still running go on without it in a smaller
    loop (Transit.mcmc_retain).  grexit=True is refused as ambiguous.  One device call's host
    arrays are bounded, the whole run's are not (see ENSEMBLE_CALL_BYTES)."""
    _check_ensemble_grexit(grtest, grexit)
    return _retrieve(transit, "demc", data, uncert, params, pmin, pmax, stepsize, numit, nchains,
                     rngs, draws, savefile, savemodel, prior=prior, priorlow=priorlow, burnin=burnin,
                     fgamma=fgamma, fepsilon=fepsilon, thinning=thinning, grtest=grtest, grexit=grexit,
                     seeds=seeds)


def _check_ensemble_grexit(grtest, grexit):
    if grexit == "each":
        if not grtest:
            raise ValueError('grexit="each" needs grtest=True: retrievals stop at the convergence '
                             'checkpoints')
    elif grexit:
        raise ValueError('grexit=True is not offered for ensembles: the retrievals converge at '
                         'different iterations; grexit="each" stops each one at its own')


def run_snooker_ensemble(transit, data, uncert, params, pmin, pmax, stepsize, numit, nchains,
                         prior=None, priorlow=None, burnin=0, thinning=1, fgamma=1.0, fepsilon=0.0,
                         hsize=1, rngs=None, draws=None, savefile=None, savemodel=None,
                         grtest=False, grexit=False, seeds=None):
    """`run_snooker` for R retrievals in one device loop (arguments as run_demc_ensemble; draws as
    snooker_draws returns them).  hsize and thinning are shared, so every retrieval's history grows
    on the same schedule.  seeds as in run_demc_ensemble.  Returns a list of R dicts with
    run_snooker's keys.  grexit="each" as in run_demc_ensemble."""
    _check_ensemble_grexit(grtest, grexit)
    return _retrieve(transit, "snooker", data, uncert, params, pmin, pmax, stepsize, numit, nchains,
                     rngs, draws, savefile, savemodel, prior=prior, priorlow=priorlow, burnin=burnin,
                     fgamma=fgamma, fepsilon=fepsilon, thinning=thinning, hsize=hsize, grtest=grtest,
                     grexit=grexit, seeds=seeds)
