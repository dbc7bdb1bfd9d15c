"""ctypes binding of libbart_b200.so (include/bart_b200.h) -- the host-side mirror of the
reference's `transit_module` interface plus the additive batched entry points.

There is no CPU path: loading fails loudly when the shared library is missing, and every
compute call fails loudly without a CUDA device (the library itself checks for sm_100).
"""
import ctypes as C
import os
import numpy as np

_trapz = getattr(np, "trapezoid", None) or np.trapz

HERE = os.path.dirname(os.path.abspath(__file__))
LIBPATH = os.environ.get("BART_B200_LIB") or os.path.join(HERE, "libbart_b200.so")   # override: A/B builds

dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int)

REJ_TGRID, REJ_TCIA, REJ_SUMQ, REJ_FEWPTS = 1, 2, 4, 8
REJ_TBOUNDS = 16        # converter: a layer outside [Tmin, Tmax] (BARTfunc.py:327-330)
REJ_ABUND = 32          # converter: the metals' abundances sum past 1 (BARTfunc.py:339-344)
REJ_NOTOOMUCH = 64
REJ_ENERGY = 128
REJ_PTMODEL = 256       # converter: PT.py refuses the parameters (BARTfunc.py:323-325)


class BartError(RuntimeError):
    pass


_lib = None


def lib():
    """Load libbart_b200.so (built in-tree by __graft_entry__.build / bart_b200/csrc/Makefile)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIBPATH):
        raise BartError("libbart_b200.so is not built (%s): run `python -c 'import "
                        "__graft_entry__ as g; g.build()'` or `make -C bart_b200/csrc`; there is "
                        "no CPU fallback" % LIBPATH)
    L = C.CDLL(LIBPATH, mode=C.RTLD_GLOBAL)
    L.transit_init.argtypes = [C.c_int, C.POINTER(C.c_char_p)]
    L.get_no_samples.restype = C.c_int
    L.get_waveno_arr.argtypes = [dp, C.c_int]
    L.set_radius.argtypes = [C.c_double]
    L.set_cloudtop.argtypes = [C.c_double]
    L.set_scattering.argtypes = [C.c_int, C.c_double]
    L.run_transit.argtypes = [dp, C.c_int, dp, C.c_int]
    L.bart_last_error.restype = C.c_char_p
    L.bart_set_batch_knobs.argtypes = [C.c_int, dp, dp, ip, dp]
    L.bart_run_batch.argtypes = [dp, C.c_int, C.c_int, dp, C.c_int, ip]
    L.bart_run_batch_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    L.bart_set_filters.argtypes = [C.c_int, ip, ip, dp, dp, C.c_double]
    L.bart_band_integrate.argtypes = [dp, C.c_int, C.c_int, dp]
    L.bart_nfilters.restype = C.c_int
    L.bart_set_energy_balance.argtypes = [C.c_int, C.c_double, C.c_double]
    L.bart_energy_balance.argtypes = [dp, C.c_int, C.c_int, ip]
    L.bart_bandflux_batch.argtypes = [dp, C.c_int, C.c_int, dp, ip]
    L.bart_bandflux_batch_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.bart_extinction_batch.argtypes = [dp, C.c_int, C.c_int, dp, C.c_int]
    L.bart_dev_alloc.restype = C.c_void_p
    L.bart_dev_alloc.argtypes = [C.c_longlong]
    L.bart_dev_free.argtypes = [C.c_void_p]
    L.bart_host_alloc_pinned.restype = C.c_void_p
    L.bart_host_alloc_pinned.argtypes = [C.c_longlong]
    L.bart_host_free_pinned.argtypes = [C.c_void_p]
    L.bart_memcpy_h2d.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong]
    L.bart_memcpy_d2h.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong]
    L.bart_timer_end.restype = C.c_double
    L.bart_kernel_stats.argtypes = [C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_longlong), dp]
    L.bart_launch_count.restype = C.c_longlong
    L.bart_grid_bytes.restype = C.c_longlong
    L.bart_debug_get.restype = C.c_longlong
    L.bart_debug_get.argtypes = [C.c_char_p, C.c_int, dp, C.c_longlong]
    L.bart_device_info.argtypes = [C.c_char_p, C.c_int, ip, ip, ip, C.POINTER(C.c_longlong),
                                   C.POINTER(C.c_longlong)]
    L.bart_comm_unique_id.argtypes = [C.c_char_p]
    L.bart_comm_init.argtypes = [C.c_int, C.c_int, C.c_char_p]
    L.bart_comm_allgather.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong]
    L.bart_bandflux_allgather_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.bart_comm_p2p.restype = C.c_int
    L.bart_build_opacity_slice.argtypes = [C.c_int, C.c_int, dp]
    L.bart_builder_stats.restype = C.c_longlong
    L.bart_builder_stats.argtypes = [C.POINTER(C.c_longlong)] * 3
    L.bart_builder_phase_ms.restype = C.c_double
    L.bart_builder_phase_ms.argtypes = [C.c_char_p]
    L.bart_line_bins.restype = C.c_longlong
    L.bart_line_bins.argtypes = [C.POINTER(C.c_longlong), C.c_longlong]
    L.bart_voigt_profile.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_float), C.c_longlong,
                                     C.POINTER(C.c_longlong)]
    L.bart_converter_init.argtypes = [C.c_int, C.c_int, dp, C.c_int, dp, dp, C.c_int, ip, C.c_int, ip,
                                      C.c_int, C.c_int, C.c_double, C.c_double, C.c_int, C.c_int,
                                      C.c_int]
    L.bart_profiles_from_params.argtypes = [dp, C.c_int, C.c_int, dp, C.c_int, ip, dp]
    L.bart_bandflux_from_params.argtypes = [dp, C.c_int, C.c_int, dp, ip]
    L.bart_bandflux_from_params_device.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.bart_chain_block.argtypes = [C.c_int, C.c_int, C.c_int, ip, ip]
    L.bart_chain_block.restype = None
    L.bart_mcmc_init.argtypes = [C.c_int, C.c_int, dp, dp, dp, dp, dp, dp, C.c_int, dp, dp,
                                 C.c_double, C.c_double, C.c_int]
    L.bart_mcmc_init_ensemble.argtypes = [C.c_int, C.c_int, C.c_int, dp, dp, dp, dp, dp, dp, C.c_int,
                                          dp, dp, C.c_double, C.c_double, C.c_int]
    L.bart_mcmc_nretr.restype = C.c_int
    L.bart_mcmc_run.argtypes = [C.c_int, dp, ip, ip, dp, dp]
    L.bart_mcmc_resume.argtypes = [C.c_int, dp]
    L.bart_mcmc_snooker_init.argtypes = [C.c_int, C.c_int, dp]
    L.bart_mcmc_run_snooker.argtypes = [C.c_int, dp, ip, ip, ip, ip, dp, ip, dp, dp]
    L.bart_mcmc_get.restype = C.c_longlong
    L.bart_mcmc_get.argtypes = [C.c_char_p, dp, C.c_longlong]
    L.bart_set_error_mode(1)
    _lib = L
    return L


def _check(rc=0):
    L = lib()
    if L.bart_error_pending() or rc != 0:
        msg = L.bart_last_error().decode(errors="replace")
        L.bart_clear_error()
        raise BartError(msg or "libbart_b200 call failed (rc=%d)" % rc)


def _d(a):
    return a.ctypes.data_as(dp)


class PinnedArray:
    """Page-locked host array (for end-to-end timing with real host<->device copies)."""

    def __init__(self, shape, dtype=np.float64):
        self.shape = tuple(np.atleast_1d(shape))
        self.dtype = np.dtype(dtype)
        n = int(np.prod(self.shape)) * self.dtype.itemsize
        self.ptr = lib().bart_host_alloc_pinned(n)
        if not self.ptr:
            raise BartError("pinned allocation of %d bytes failed" % n)
        buf = (C.c_char * n).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype).reshape(self.shape)

    def free(self):
        if self.ptr:
            self.array = None
            lib().bart_host_free_pinned(self.ptr)
            self.ptr = None


class Transit:
    """One transit instance per process, like the reference (transit.c:7-12)."""

    def __init__(self, cfg=None, argv=None, device=None):
        L = lib()
        if device is not None:
            _check(L.bart_set_device(int(device)))
        if argv is None:
            argv = ["transit", "-c", cfg]
        args = [a.encode() if isinstance(a, str) else a for a in argv]
        arr = (C.c_char_p * (len(args) + 1))(*args, None)
        L.transit_init(len(args), arr)
        _check()
        self.nwave = L.get_no_samples()
        self.nlayer = L.bart_nlayers()
        self.nspec = L.bart_nspecies()
        self.n_in = (self.nspec + 1) * self.nlayer
        self.eclipse = bool(L.bart_is_eclipse())
        self.nfilters = 0

    # ---- the reference surface ----
    def get_no_samples(self):
        return lib().get_no_samples()

    def get_waveno_arr(self, n=None):
        n = self.nwave if n is None else n
        out = np.zeros(n)
        lib().get_waveno_arr(_d(out), n)
        return out

    def set_radius(self, r):
        lib().set_radius(float(r))

    def set_cloudtop(self, c):
        lib().set_cloudtop(float(c))

    def set_scattering(self, flag, v):
        lib().set_scattering(int(flag), float(v))

    def run_transit(self, profiles, nwave=None):
        nwave = self.nwave if nwave is None else nwave
        p = np.ascontiguousarray(profiles, dtype=np.float64).ravel()
        out = np.zeros(nwave)
        lib().run_transit(_d(p), p.size, _d(out), nwave)
        _check()
        return out

    def free_memory(self):
        lib().free_memory()
        _check()

    # ---- additive ----
    def set_batch_knobs(self, nmodels, refradius=None, cloudtop=None, scat_flag=None,
                        scat_logext=None):
        def arr(x, dt):
            return None if x is None else np.ascontiguousarray(x, dtype=dt)
        r, c, f, s = arr(refradius, np.float64), arr(cloudtop, np.float64), \
            arr(scat_flag, np.int32), arr(scat_logext, np.float64)
        _check(lib().bart_set_batch_knobs(
            int(nmodels), None if r is None else _d(r), None if c is None else _d(c),
            None if f is None else f.ctypes.data_as(ip), None if s is None else _d(s)))

    def run_batch(self, profiles, out=None, status=None):
        p = np.ascontiguousarray(profiles, dtype=np.float64)
        if p.ndim == 1:
            p = p[None, :]
        M = p.shape[0]
        if out is None:
            out = np.empty((M, self.nwave))
        if status is None:
            status = np.zeros(M, dtype=np.int32)
        _check(lib().bart_run_batch(_d(p), M, p.shape[1], _d(out), self.nwave,
                                    status.ctypes.data_as(ip)))
        return out, status

    def set_filters(self, start, count, weight, star=None, rprs=1.0):
        start = np.ascontiguousarray(start, dtype=np.int32)
        count = np.ascontiguousarray(count, dtype=np.int32)
        weight = np.ascontiguousarray(weight, dtype=np.float64)
        st = None if star is None else np.ascontiguousarray(star, dtype=np.float64)
        _check(lib().bart_set_filters(len(start), start.ctypes.data_as(ip),
                                      count.ctypes.data_as(ip), _d(weight),
                                      None if st is None else _d(st), float(rprs)))
        self.nfilters = len(start)

    def set_energy_balance(self, tstar, rstar_m, sma_m, rplanet_m, on=True):
        """Switch on BARTfunc's energy-balance rejection (code/BARTfunc.py:366-383; arguments as it
        reads them from the TEP file: Ts [K], Rs, a, Rp [m]) for every band-flux call."""
        sig, j2erg = 5.670367e-8, 1e7                      # code/constants.py:19, BARTfunc.py:375
        e_in = sig * tstar ** 4 * rstar_m ** 2 * np.pi * rplanet_m ** 2 / sma_m ** 2 * j2erg
        _check(lib().bart_set_energy_balance(1 if on else 0, float(e_in), float(4 * (rplanet_m * 100) ** 2)))
        return e_in

    def energy_balance(self, spectra):
        s = np.ascontiguousarray(np.atleast_2d(spectra), dtype=np.float64)
        out = np.zeros(s.shape[0], dtype=np.int32)
        _check(lib().bart_energy_balance(_d(s), s.shape[0], s.shape[1], out.ctypes.data_as(ip)))
        return out

    def band_integrate(self, spectra):
        s = np.ascontiguousarray(spectra, dtype=np.float64)
        if s.ndim == 1:
            s = s[None, :]
        out = np.empty((s.shape[0], self.nfilters))
        _check(lib().bart_band_integrate(_d(s), s.shape[0], s.shape[1], _d(out)))
        return out

    def bandflux_batch(self, profiles, out=None, status=None):
        p = np.ascontiguousarray(profiles, dtype=np.float64)
        if p.ndim == 1:
            p = p[None, :]
        M = p.shape[0]
        if out is None:
            out = np.empty((M, self.nfilters))
        if status is None:
            status = np.zeros(M, dtype=np.int32)
        _check(lib().bart_bandflux_batch(_d(p), M, p.shape[1], _d(out),
                                         status.ctypes.data_as(ip)))
        return out, status

    def extinction_batch(self, profiles, total=False, fetch=True):
        p = np.ascontiguousarray(profiles, dtype=np.float64)
        if p.ndim == 1:
            p = p[None, :]
        M = p.shape[0]
        out = np.empty((M, self.nlayer, self.nwave)) if fetch else None
        _check(lib().bart_extinction_batch(_d(p), M, p.shape[1],
                                           None if out is None else _d(out), 1 if total else 0))
        return out

    # ---- retrieval loop on the device (include/bart_b200.h part 3) -------------------------
    PT_TYPES = {"iso": 0, "line": 1, "adiabatic": 2, "madhu_noinv": 3, "madhu_inv": 4, "piette": 5}
    PT_NPARS = {"iso": 1, "line": 5, "adiabatic": 3, "madhu_noinv": 5, "madhu_inv": 6, "piette": 8}

    def converter_init(self, pressure_bar, species, abundances, molfit, pt_type="line", pt_args=None,
                       tint_type="const", tmin=400.0, tmax=3000.0, nrad=None, ncloud=0, nray=0):
        """Input-converter set-up of code/BARTfunc.py:139-222: `abundances[layer][species]`,
        `pressure_bar[layer]` and `species` as makeatm.readatm returns them; `molfit` the fitted
        molecule names; pt_type one of BARTfunc.py:150-155's names; pt_args = (R_star, T_star, T_int,
        sma, gravity) for PT_line."""
        species = list(species)
        press = np.ascontiguousarray(pressure_bar, dtype=np.float64)
        ab = np.ascontiguousarray(abundances, dtype=np.float64)
        if ab.shape != (self.nlayer, self.nspec) or press.shape != (self.nlayer,):
            raise BartError("abundances must be [%d layers][%d species]" % (self.nlayer, self.nspec))
        imol = np.array([species.index(m) for m in molfit], dtype=np.int32)
        imetals = np.array([i for i, s in enumerate(species) if s not in ("H2", "He", "H-", "e-")],
                           dtype=np.int32)
        npt = self.PT_NPARS[pt_type]
        if nrad is None:
            nrad = 0 if self.eclipse else 1
        args = np.ascontiguousarray(pt_args if pt_args is not None else np.zeros(5), dtype=np.float64)
        _check(lib().bart_converter_init(self.PT_TYPES[pt_type], npt, _d(args),
                                         int(tint_type == "thorngren"), _d(press), _d(ab), len(imol),
                                         imol.ctypes.data_as(ip), len(imetals),
                                         imetals.ctypes.data_as(ip), species.index("H2"),
                                         species.index("He"), float(tmin), float(tmax), int(nrad),
                                         int(ncloud), int(nray)))
        self.npars = lib().bart_converter_npars()
        return self.npars

    def profiles_from_params(self, params):
        """params[M][npars] -> (profiles[M][n_in], status[M], knobs[3][M]) (parity/debug)."""
        params = np.ascontiguousarray(np.atleast_2d(params), dtype=np.float64)
        M = params.shape[0]
        prof = np.zeros((M, self.n_in))
        status = np.zeros(M, dtype=np.int32)
        knobs = np.zeros((3, M))
        _check(lib().bart_profiles_from_params(_d(params), M, params.shape[1], _d(prof), self.n_in,
                                               status.ctypes.data_as(ip), _d(knobs)))
        return prof, status, knobs

    def bandflux_from_params(self, params, out=None, status=None):
        """One BARTfunc.py worker iteration (309-399) for a batch of proposals."""
        params = np.ascontiguousarray(np.atleast_2d(params), dtype=np.float64)
        M = params.shape[0]
        if out is None:
            out = np.empty((M, self.nfilters))
        if status is None:
            status = np.zeros(M, dtype=np.int32)
        _check(lib().bart_bandflux_from_params(_d(params), M, params.shape[1], _d(out),
                                               status.ctypes.data_as(ip)))
        return out, status

    def mcmc_init(self, params, pmin, pmax, stepsize, data, uncert, prior=None, priorlow=None,
                  fgamma=1.0, fepsilon=0.0, burnin=0):
        params = np.ascontiguousarray(np.atleast_2d(params), dtype=np.float64)
        nchains, npars = params.shape
        f = lambda a: np.ascontiguousarray(a if a is not None else np.zeros(npars), dtype=np.float64)
        pmin, pmax, stepsize, prior, priorlow = (f(a) for a in (pmin, pmax, stepsize, prior, priorlow))
        data = np.ascontiguousarray(data, dtype=np.float64)
        uncert = np.ascontiguousarray(uncert, dtype=np.float64)
        _check(lib().bart_mcmc_init(nchains, npars, _d(params), _d(pmin), _d(pmax), _d(stepsize),
                                    _d(prior), _d(priorlow), len(data), _d(data), _d(uncert),
                                    float(fgamma), float(fepsilon), int(burnin)))
        self._mc_shape = (nchains, npars, int(np.sum(stepsize > 0)), len(data))
        self._mc_ensemble = False

    def mcmc_init_ensemble(self, params, pmin, pmax, stepsize, data, uncert, prior=None,
                           priorlow=None, fgamma=1.0, fepsilon=0.0, burnin=0):
        """R independent retrievals in one device loop (bart_mcmc_init_ensemble): params[R][C][P]
        starting points, data / uncert[R][D]; bounds, step sizes and priors shared.  Afterwards the
        mcmc_* calls take and return every array behind a leading [R] axis."""
        params = np.ascontiguousarray(params, dtype=np.float64)
        if params.ndim != 3:
            raise BartError("params must be [retrievals][chains][parameters]")
        nretr, nchains, npars = params.shape
        f = lambda a: np.ascontiguousarray(a if a is not None else np.zeros(npars), dtype=np.float64)
        pmin, pmax, stepsize, prior, priorlow = (f(a) for a in (pmin, pmax, stepsize, prior, priorlow))
        data = np.ascontiguousarray(data, dtype=np.float64)
        uncert = np.ascontiguousarray(uncert, dtype=np.float64)
        if data.ndim != 2 or data.shape[0] != nretr or uncert.shape != data.shape:
            raise BartError("data and uncert must be [%d retrievals][data points]" % nretr)
        _check(lib().bart_mcmc_init_ensemble(nretr, nchains, npars, _d(params), _d(pmin), _d(pmax),
                                             _d(stepsize), _d(prior), _d(priorlow), data.shape[1],
                                             _d(data), _d(uncert), float(fgamma), float(fepsilon),
                                             int(burnin)))
        self._mc_shape = (nchains, npars, int(np.sum(stepsize > 0)), data.shape[1])
        self._mc_ensemble = True

    def _mc_lead(self):
        """Leading axis of the loop's arrays: () after mcmc_init, (R,) after mcmc_init_ensemble."""
        return (lib().bart_mcmc_nretr(),) if getattr(self, "_mc_ensemble", False) else ()

    def _mc_refuse(self, lead, what):
        raise BartError("%s do not have MC3's shapes for %s%d chains" % (
            what, "%d retrievals x " % lead[0] if lead else "", self._mc_shape[0]))

    def mcmc_resume(self, nold, curmodel=None):
        """MC3's resume=True (mcmc.py:254-269) after mcmc_init with the old run's last states."""
        if curmodel is not None:
            curmodel = np.ascontiguousarray(curmodel, dtype=np.float64)
            nchains, npars, nfree, ndata = self._mc_shape
            lead = self._mc_lead()
            if curmodel.shape != lead + (nchains, ndata):
                raise BartError("curmodel must be [%s%d chains][%d data]"
                                % ("%d retrievals][" % lead[0] if lead else "", nchains, ndata))
        _check(lib().bart_mcmc_resume(int(nold), None if curmodel is None else _d(curmodel)))

    def mcmc_run(self, support, r1, r2, unif, ugamma):
        support = np.ascontiguousarray(support, dtype=np.float64)
        unif = np.ascontiguousarray(unif, dtype=np.float64)
        ugamma = np.ascontiguousarray(ugamma, dtype=np.float64)
        r1 = np.ascontiguousarray(r1, dtype=np.int32)
        r2 = np.ascontiguousarray(r2, dtype=np.int32)
        lead = self._mc_lead()
        niter = unif.shape[-2] if unif.ndim >= 2 else 0
        nchains, npars, nfree, ndata = self._mc_shape
        if support.shape != lead + (niter, nchains, nfree) or r1.shape != lead + (nchains, niter) or \
                r2.shape != lead + (nchains, niter) or unif.shape != lead + (niter, nchains) or \
                ugamma.shape != lead + (niter, nchains):
            if not lead:
                raise BartError("random streams do not have MC3's shapes for %d chains x %d iterations"
                                % (nchains, niter))
            self._mc_refuse(lead, "random streams")
        _check(lib().bart_mcmc_run(niter, _d(support), r1.ctypes.data_as(ip), r2.ctypes.data_as(ip),
                                   _d(unif), _d(ugamma)))
        self._mc_niter = niter

    def mcmc_snooker_init(self, z0, thinning=1):
        """z0[hsize][nchains][nfree] ([R][hsize][nchains][nfree] for an ensemble): MC3's M0 initial
        history samples (mcmc.py:421-424)."""
        nchains, npars, nfree, ndata = self._mc_shape
        lead = self._mc_lead()
        z0 = np.ascontiguousarray(z0, dtype=np.float64)
        if z0.ndim != 3 + len(lead) or z0.shape[:len(lead)] != lead or z0.shape[-2:] != (nchains, nfree):
            raise BartError("z0 must be [%shsize][%d][%d]" % ("%d][" % lead[0] if lead else "", nchains, nfree))
        hsize = z0.shape[len(lead)]
        _check(lib().bart_mcmc_snooker_init(hsize, int(thinning), _d(z0)))
        self._mc_zsize, self._mc_thinning = hsize, int(thinning)

    def mcmc_run_snooker(self, support, i1, i2, iz, ic, usnooker, usn_offset, unif, ugamma):
        """Streams of run_snooker's shapes; for an ensemble each behind [R], usnooker the
        retrievals' factor rows one after the other and usn_offset[R][niter+1] absolute rows."""
        nchains, npars, nfree, ndata = self._mc_shape
        lead = self._mc_lead()
        support, unif, ugamma, usnooker = (np.ascontiguousarray(a, dtype=np.float64)
                                           for a in (support, unif, ugamma, usnooker))
        i1, i2, iz, ic, usn_offset = (np.ascontiguousarray(a, dtype=np.int32)
                                      for a in (i1, i2, iz, ic, usn_offset))
        niter = unif.shape[-2] if unif.ndim >= 2 else 0
        if support.shape != lead + (niter, nchains, nfree) or ugamma.shape != lead + (niter, nchains) or \
                unif.shape != lead + (niter, nchains) or \
                any(a.shape != lead + (niter, nchains) for a in (i1, i2, iz, ic)) or \
                usn_offset.shape != lead + (niter + 1,) or \
                usnooker.shape != (usn_offset.flat[-1] if usn_offset.size else -1, nfree):
            if not lead:
                raise BartError("random streams do not have MC3's shapes for %d chains x %d iterations"
                                % (nchains, niter))
            self._mc_refuse(lead, "snooker streams")
        _check(lib().bart_mcmc_run_snooker(
            niter, _d(support), i1.ctypes.data_as(ip), i2.ctypes.data_as(ip), iz.ctypes.data_as(ip),
            ic.ctypes.data_as(ip), _d(usnooker), usn_offset.ctypes.data_as(ip), _d(unif), _d(ugamma)))
        self._mc_niter = niter
        self._mc_zsize += len(range(0, niter, self._mc_thinning)) + 1     # upper bound, see mcmc_get

    def mcmc_get(self, name):
        nchains, npars, nfree, ndata = self._mc_shape
        lead = self._mc_lead()
        if name in ("Z", "Zchisq"):
            # _mc_zsize is an upper bound (it counts thinned rows per call; the library grows Z on
            # the GLOBAL iteration number, like MC3): size the result from what the library returns
            tail = (nchains, npars) if name == "Z" else (nchains,)
            out = np.zeros(lead + (getattr(self, "_mc_zsize", 0),) + tail)
            n = lib().bart_mcmc_get(name.encode(), _d(out), out.size)
            _check(0 if n >= 0 else -1)
            rows = n // (int(np.prod(lead + tail)))
            if not lead:
                return out[:rows]
            return out.ravel()[:n].reshape(lead + (rows,) + tail).copy()
        shapes = {"allparams": (nchains, nfree, getattr(self, "_mc_niter", 0)),
                  "allmodel": (nchains, ndata, getattr(self, "_mc_niter", 0)),
                  "params": (nchains, npars), "currchisq": (nchains,), "numaccept": (nchains,),
                  "outbounds": (nchains, nfree), "bestp": (npars,), "bestchisq": (1,),
                  "bestmodel": (ndata,), "models": (nchains, ndata)}
        shape = lead + shapes[name] if name != "bestchisq" or not lead else lead
        out = np.zeros(shape)
        n = lib().bart_mcmc_get(name.encode(), _d(out), out.size)
        _check(0 if n >= 0 else -1)
        return out

    def debug_keep(self, on=True):
        lib().bart_debug_keep(1 if on else 0)

    def debug_get(self, name, model=0, n=None):
        cap = n if n is not None else max(self.nwave * self.nlayer, 64 * self.nlayer)
        out = np.zeros(cap)
        got = lib().bart_debug_get(name.encode(), model, _d(out), cap)
        _check(0 if got >= 0 else -1)
        return out[:got]


# ---- module-level helpers ----
def bind_to_device_numa(device):
    """Pin this process to the CPU cores NVML reports as local to GPU `device` (what `numactl` /
    `mpirun --bind-to` do for a one-process-per-GPU job).  Call it before the library is
    initialised: pinned host buffers then come from the GPU's own NUMA node and 8 ranks do not
    funnel their host copies through one socket.  Returns the CPU list, or None when NVML or the
    affinity call is not available (nothing changes then)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(device))
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:
        return None


def device_info():
    name = C.create_string_buffer(256)
    sm, ma, mi = C.c_int(), C.c_int(), C.c_int()
    l2, hbm = C.c_longlong(), C.c_longlong()
    _check(lib().bart_device_info(name, 256, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(l2),
                                  C.byref(hbm)))
    return dict(name=name.value.decode(), sm_count=sm.value, cc=(ma.value, mi.value),
                l2_bytes=l2.value, hbm_bytes=hbm.value)


def kernel_stats():
    out = {}
    i = 0
    while True:
        name = C.create_string_buffer(128)
        n, ms = C.c_longlong(), C.c_double()
        if lib().bart_kernel_stats(i, name, 128, C.byref(n), C.byref(ms)) != 0:
            break
        out[name.value.decode()] = dict(launches=n.value, ms=ms.value)
        i += 1
    return out


def read_kurucz(kfile, temperature, logg):
    """Stellar spectrum of the Kurucz grid model nearest to (temperature, logg): what
    code/wine.py:69-124 `readkurucz` returns through code/kurucz_inten.py:162-318 -- (starfl [erg s-1
    cm-2 cm], starwn [cm-1] ascending, model temperature, model log g).  File layout: a FORTRAN
    reader as preamble ending in a line `END`, the wavelength table (nm, 10-character fields), then
    per model a `TEFF ... GRAVITY ...` line, the line-blanketed Eddington fluxes and the continuum
    fluxes (10-character fields, erg cm-2 s-1 Hz-1 sr-1).  Only the selected model is parsed."""
    c_light = 299792458.0                                     # scipy.constants.c
    with open(kfile, "r") as f:
        lines = f.read().replace("\r", "\n").split("\n")
    heads = [i for i, ln in enumerate(lines) if ln.startswith("TEFF")]
    temp = np.array([float(lines[i][5:12]) for i in heads])
    grav = np.array([float(lines[i][22:29]) for i in heads])
    start = max(i for i, ln in enumerate(lines[:heads[0]]) if ln.endswith("END")) + 1
    fields = lambda block: [float(block[j:j + 10]) for j in range(0, len(block), 10) if block[j:j + 10].strip()]
    wave = np.array(fields("".join(lines[start:heads[0]])))
    wave = wave[wave != 0] * 1e-9                             # nm -> m
    nline = (heads[2] - heads[1] - 1) // 2
    tmodel = temp[np.argmin(np.abs(temp - temperature))]
    gmodel = grav[np.argmin(np.abs(grav - logg))]
    imodel = np.where((temp == tmodel) & (grav >= gmodel))[0][0]
    h = heads[imodel]
    inten = np.zeros(wave.size)
    vals = fields("".join(lines[h + 1:h + 1 + nline]))
    inten[:len(vals)] = vals[:wave.size]
    inten *= 4.0 * 1e-3                                       # Eddington flux -> brightness, cgs -> MKS
    freq = np.flipud(c_light / wave)
    inten = inten[::-1]
    starwn = freq / c_light * 1e-2
    starfl = inten * 1e3 * np.pi * (1e2 * c_light)            # per Hz -> per cm-1, MKS -> cgs, sr-1 -> flux
    return starfl, starwn, tmodel, gmodel


def filters_from_files(specwn, filter_files, starwn=None, starfl=None):
    """Host-side precompute of stage (c): the same resampling BARTfunc.py:245-291 does with
    wine.readfilter / wine.resample (linear interpolation of filter and stellar spectrum onto the
    spectrum grid inside the filter span, filter normalised to unit trapezoid integral).
    Returns (start, count, weight_concat, star_concat|None)."""
    starts, counts, weights, stars = [], [], [], []
    for path in filter_files:
        with open(path) as f:
            lines = f.readlines()
        while lines[0].startswith("#") or not lines[0].strip():
            lines.pop(0)
        wl = np.array([float(l.split()[0]) for l in lines])
        tr = np.array([float(l.split()[1]) for l in lines])
        fwn, ftr = (1.0 / (wl * 1e-4))[::-1], tr[::-1]
        idx = np.where((specwn < fwn[-1]) & (fwn[0] < specwn))[0]
        if len(idx) < 2 or np.any(np.diff(idx) != 1):
            raise BartError("filter %s does not map to a contiguous spectrum range" % path)
        ifilt = np.interp(specwn[idx], fwn, ftr)
        nif = ifilt / _trapz(ifilt, specwn[idx])
        starts.append(idx[0])
        counts.append(len(idx))
        weights.append(nif)
        if starwn is not None:
            stars.append(np.interp(specwn[idx], starwn, starfl))
    star = np.concatenate(stars) if stars else None
    return (np.array(starts, dtype=np.int32), np.array(counts, dtype=np.int32),
            np.concatenate(weights), star)
