/* bart_b200.h -- C ABI of libbart_b200.so: the B200-native `transit` forward model.
 *
 * Plain C, pointers + sizes only.  Part 1 is the reference's own boundary, same names,
 * argument meaning and units, so the existing SWIG/ctypes/cgo binding of BART's `transit`
 * binds this library unchanged.  Part 2 is additive (batched evaluation, band integration,
 * multi-GPU exchange, timing, introspection); nothing in part 1 depends on it being called.
 *
 * Reference citations are into exosports/BART, modules/transit/transit/.
 * One instance per process (the reference keeps one global `struct transit`, src/transit.c:7-12).
 * All arithmetic is fp64.  There is no CPU fallback: every entry point that computes needs a
 * CUDA device of compute capability 10.0 and fails loudly without one.
 */
#ifndef BART_B200_H
#define BART_B200_H

#ifdef __cplusplus
extern "C" {
#endif

/* ===================================================================================== */
/* Part 1 -- the reference boundary (src/transit.c:14-22, include/transit.h:44-49,
 *           SWIG surface src/transit.i:12-31)                                            */

/* replaces transit_init (src/transit.c:25-74): parse `argv` (["transit","-c",cfgfile,...],
 * option table of src/argum.c:112-320, `key value` file grammar of pu/src/procopt.c:649-704),
 * read atmosphere / molecules / TLI header / CIA files, read -- or, when the named opacity
 * file does not exist, BUILD (Voigt line-by-line, src/opacity.c:218-427) and write -- the
 * opacity grid, and make everything resident in HBM.  Without an `opacityfile` key the
 * reference keeps only the Voigt table (src/opacity.c:28-36) and computes every layer's
 * extinction line by line inside tau() (src/tau.c:163-175,253-264 -> computemolext with
 * permol = 0, src/extinction.c:281-529): same here, the TLI lines and the Voigt table are made
 * resident and every run_transit / bart_run_batch call evaluates its (model, layer) cells with
 * the builder kernels at the layers' own temperatures.  A model's table is staged whole in
 * the shared memory of one block, so the layer count is bounded by the device: a configuration
 * with more layers than its geometry, molecule and CIA counts allow is refused here, with that
 * limit in the message.                                                                   */
void transit_init(int argc, char **argv);

/* replaces get_no_samples (src/transit.c:77-80): number of spectrum wavenumbers.         */
int get_no_samples(void);

/* replaces get_waveno_arr (src/transit.c:82-95): wavenumber grid in cm-1; -1 fill when not
 * initialised, like the reference.                                                       */
void get_waveno_arr(double *waveno_arr, int waveno);

/* replaces set_radius (src/transit.c:98-100): reference radius r0, units of the atmosphere
 * file's radius factor (km for TEA files); applies to subsequent models.                 */
void set_radius(double refradius);

/* replaces set_cloudtop (src/transit.c:103-109): opaque cloud deck, log10(bar).          */
void set_cloudtop(double cloudtop);

/* replaces set_scattering (src/transit.c:112-115): flag 1 = Lecavelier (logext), 2 = polar. */
void set_scattering(int flag, double scattering);

/* replaces run_transit (src/transit.c:118-122): one forward model.
 * re_input[(1+nspecies)*nlayers] = [T(layers) | q_species0(layers) | ...], layers bottom ->
 * top in atmosphere-file order (src/readatm.c:735-744); transit_out[nwave] receives the
 * emergent flux (eclipse, erg s-1 cm-1) or the modulation (transit, (Rp/Rs)^2).
 * With `savefiles yes` in the configuration (src/tau.c:179-190,308-329) the call also writes
 * tau.dat, CIA.dat, mol_extion.dat, total_extion.dat, cloud_extion.dat and scatt_extion.dat
 * into the working directory in the reference's text layouts (src/tau.c:360-518); tau.dat
 * is what code/cf.py:68-135 reads for the contribution functions.                        */
void run_transit(double *re_input, int transint, double *transit_out, int transit_out_size);

/* replaces free_memory (src/transit.c:216-228).                                          */
void free_memory(void);

/* ===================================================================================== */
/* Part 2 -- additive entry points                                                         */

#define BART_OK 0

/* Error handling.  The reference prints and exit()s on any failure (include/transit.h:91-98).
 * mode 0 (default) reproduces that for the part-1 functions; mode 1 makes every function
 * return, leaving a message for bart_last_error (the Python module uses mode 1).         */
void        bart_set_error_mode(int mode);
const char *bart_last_error(void);
int         bart_error_pending(void);
void        bart_clear_error(void);

/* Device selection; call before transit_init (default: $BART_DEVICE, else $LOCAL_RANK, else 0). */
int  bart_set_device(int ordinal);
int  bart_get_device(void);
int  bart_device_info(char *name, int name_len, int *sm_count, int *cc_major, int *cc_minor,
                      long long *l2_bytes, long long *hbm_bytes);

/* Shapes after transit_init.                                                              */
int  bart_nlayers(void);
int  bart_nspecies(void);
int  bart_ngridmol(void);
int  bart_ngridtemp(void);
int  bart_is_eclipse(void);
long long bart_grid_bytes(void);

/* Batched forward model.  profiles[nmodels][n_in] (same per-model layout as run_transit),
 * spectra[nmodels][n_out].  Host pointers; the call copies in, computes and copies out.
 * status[nmodels] (may be NULL) receives 0 or a rejection code per model (BART_REJ_*)
 * instead of the reference's exit(): the spectrum of a rejected model is filled with -1.   */
int  bart_run_batch(const double *profiles, int nmodels, int n_in, double *spectra, int n_out,
                    int *status);
#define BART_REJ_TGRID   1   /* a layer temperature outside the opacity-grid range          */
#define BART_REJ_TCIA    2   /* outside a CIA table's range (src/crosssec.c:293-309)        */
#define BART_REJ_SUMQ    4   /* sum of abundances > 1.001 (src/readatm.c:152-156)           */
#define BART_REJ_FEWPTS  8   /* transit: fewer than 3 points for the modulation integral    */
#define BART_REJ_NOTOOMUCH 64 /* transit, modlevel -1: tau never reached toomuch at some
                                wavenumber (src/slantpath.c:308-316,458-460)                  */

/* Per-model knobs for the batched calls (the reference's setters are per-process state that
 * BARTfunc.py sets before each run_transit, code/BARTfunc.py:350-360).  Any pointer may be
 * NULL to keep the process-wide value; arrays have nmodels entries.                       */
int  bart_set_batch_knobs(int nmodels, const double *refradius, const double *cloudtop,
                          const int *scat_flag, const double *scat_logext);

/* Same, with device-resident buffers (for callers that keep proposals on the GPU).        */
int  bart_run_batch_device(const double *d_profiles, int nmodels, int n_in, double *d_spectra,
                           int n_out, int *d_status);

/* Stage (c): band integration (code/wine.py:127-199, code/BARTfunc.py:386-396).
 * nfilters filters; filter f covers spectrum samples [start[f], start[f]+count[f]);
 * weight[] and star[] are the concatenated per-sample normalised filter transmission and
 * stellar flux (star may be NULL: no division, `transit`/`direct` modes); rprs = Rp/Rs.    */
int  bart_set_filters(int nfilters, const int *start, const int *count, const double *weight,
                      const double *star, double rprs);
int  bart_nfilters(void);            /* filters configured by bart_set_filters (0 before) */
/* Energy-balance rejection (code/BARTfunc.py:366-383), applied by every call that returns band
 * fluxes once switched on: a model with trapz(spectrum, wn) * out_scale > e_in is rejected
 * (BART_REJ_ENERGY, band fluxes -1).  The caller computes e_in = sigma Ts^4 Rs^2 pi Rp^2 / a^2 * 1e7
 * and out_scale = 4 (100 Rp)^2 (Rp in m) like BARTfunc does.
 * bart_energy_balance applies the test to host spectra[nmodels][nwave] (rejected[m] = 0 or
 * BART_REJ_ENERGY): the kernel on its own, for parity tests.                                     */
int  bart_set_energy_balance(int on, double e_in, double out_scale);
int  bart_energy_balance(const double *spectra, int nmodels, int nwave, int *rejected);
int  bart_band_integrate(const double *spectra, int nmodels, int nwave, double *bandflux);
/* profiles -> band fluxes in one call; spectra never leave the device.
 * bandflux[nmodels][nfilters]; rejected models get -1 in every band (BARTfunc.py:327-330).  */
int  bart_bandflux_batch(const double *profiles, int nmodels, int n_in, double *bandflux,
                         int *status);
int  bart_bandflux_batch_device(const double *d_profiles, int nmodels, int n_in,
                                double *d_bandflux, int *d_status);

/* Stand-alone opacity lookup (src/extinction.c:534-581 + the sum of src/tau.c:231-232):
 * materialises ext[nmodels][nlayer][nwave] on the device (debug/roofline use).            */
int  bart_extinction_batch(const double *profiles, int nmodels, int n_in, double *ext_out,
                           int what /*0 molecular, 1 total incl. CIA/scattering/cloud, 2 CIA only*/);

/* Device memory helpers for callers without a CUDA runtime of their own.                  */
void *bart_dev_alloc(long long bytes);
void  bart_dev_free(void *p);
void *bart_host_alloc_pinned(long long bytes);
void  bart_host_free_pinned(void *p);
int   bart_memcpy_h2d(void *dst, const void *src, long long bytes);
int   bart_memcpy_d2h(void *dst, const void *src, long long bytes);
int   bart_sync(void);

/* Timing on the library's own stream (CUDA events).  bart_timer_begin/end bracket a region
 * and return milliseconds; with profiling on, every kernel launch is bracketed too and
 * bart_kernel_stats reports, per kernel name, launches and total milliseconds.             */
int    bart_timer_begin(void);
double bart_timer_end(void);
void   bart_profile_enable(int on);
void   bart_profile_reset(void);
int    bart_kernel_stats(int index, char *name, int name_len, long long *launches, double *ms);
long long bart_launch_count(void);
int    bart_flush_l2(void);

/* Introspection for parity tests: copy an intermediate of the LAST batched call to host.
 * names: "radius","density","temp","tau","last","cia","ext","simpson"...; returns the number
 * of doubles written or <0.                                                                */
long long bart_debug_get(const char *name, int model, double *out, long long capacity);
void      bart_debug_keep(int on);   /* keep tau/last columns of the next calls (costs HBM) */

/* Multi-GPU: one process per GPU; chains are partitioned by rank and each generation ends with
 * one all-gather of [nlocal][width] doubles (replaces the MPI Scatter/Gather of
 * modules/MCcubed/MCcubed/mc/mcmc.py:583-585 / code/BARTfunc.py:312,399).                   */
int  bart_comm_unique_id(char *id128);
int  bart_comm_init(int rank, int world, const char *id128);
int  bart_comm_allgather(const double *d_send, double *d_recv, long long count_per_rank);
int  bart_comm_finalize(void);
/* Fused band integration + all-gather.  bart_comm_init also maps a small window of every peer
 * GPU through CUDA IPC (NVLink/NVSwitch peer memory); when that succeeded on every rank
 * (bart_comm_p2p() == 1; $BART_P2P=0 disables it) the band-integration kernel stores each band
 * flux directly into all ranks' windows and releases a per-rank arrival flag, and a one-CTA
 * consumer kernel waits for the flags -- no NCCL call on the per-generation path.  Used by the
 * device-resident retrieval loop (part 3) and by:
 * forward models of this rank's `nmodels` proposals -> d_bandflux[nmodels][nfilters] and every
 * rank's block in d_all[world][nmodels][nfilters] (same nmodels on every rank); falls back to
 * ncclAllGather when the windows are unavailable or too small.                             */
int  bart_comm_p2p(void);
int  bart_bandflux_allgather_device(const double *d_profiles, int nmodels, int n_in,
                                    double *d_bandflux, double *d_all);

/* Opacity-grid builder (--justOpacity; src/opacity.c:218-427, src/extinction.c:281-529,
 * pu/src/voigt.c).  transit_init builds the grid itself when the file is missing; these expose
 * the pieces: t_begin/t_end select a slice of the temperature axis (T-sharded multi-GPU build). */
int  bart_build_opacity_slice(int t_begin, int t_end, double *host_out /*[layer][t][mol][wn]*/);
long long bart_builder_stats(long long *nlines, long long *ngroups, long long *neval);
/* milliseconds spent so far in a build phase: "read_tli_host", "grouping_host", "voigt_table",
 * "kmax", "strength", "widths", "accumulate", "d2h" (CUDA events on the build stream).      */
double bart_builder_phase_ms(const char *name);
long long bart_line_bins(long long *iown_out, long long capacity);  /* bit-exact bin trace   */
int  bart_voigt_profile(int idop, int ilor, float *out, long long capacity, long long *halfsize);

/* ===================================================================================== */
/* Part 3 -- the retrieval loop around the forward model, on the device (additive).
 * In the reference these run in Python on the host, once per proposal and per chain:
 * code/BARTfunc.py:309-399 (one MPI worker per chain) and modules/MCcubed/MCcubed/mc/mcmc.py.
 * One loop holds an ensemble of independent retrievals (bart_mcmc_init_ensemble); between run
 * calls bart_mcmc_retain shrinks it to the retrievals still running, which is how the driver
 * stops each retrieval at its own MC3 convergence checkpoint (driver.py, grexit="each").        */

#define BART_REJ_TBOUNDS 16  /* temperature profile outside [Tmin, Tmax] (BARTfunc.py:327-330)   */
#define BART_REJ_ABUND   32  /* sum of metal abundances > 1 (BARTfunc.py:339-344)                */
#define BART_REJ_ENERGY  128 /* energy balance failed: E_out > E_in (BARTfunc.py:366-383)            */
#define BART_REJ_PTMODEL 256 /* Madhusudhan-Seager parameters the reference's PT.py refuses (negative
                                boundary temperatures, code/PT.py:337-340,543-545)                  */

/* replaces the input-converter set-up of code/BARTfunc.py:139-222.
 * pt_type: 0 PT_iso (1 parameter), 1 PT_line (5: log kappa, log gamma1, log gamma2, alpha, beta;
 * code/PT.py:589-697), 2 PT_adiabatic (3; PT.py:741-750), 3 PT_NoInversion (5: a1 a2 p1 p3 T3;
 * PT.py:384-586), 4 PT_Inversion (6: a1 a2 p1 p2 p3 T3; PT.py:157-377), 5 PT_piette (8: T0 and seven
 * temperature steps; PT.py:752-812).  Models 3-5 smooth over the layers with
 * scipy.ndimage.gaussian_filter1d(mode='nearest'), restated on the device (sigma 4 layers, or 0.3 dex
 * for PT_piette, whose pressure grid must be uniform in log p and separate the eight node layers).
 * pt_args[5] = {R_star m, T_star K,
 * T_int K, sma m, gravity cm s-2} for PT_line (BARTfunc.py:206-211); tint_thorngren != 0 computes
 * T_int after Thorngren et al. 2019 (PT.py:671-676).  pressure_bar[nlayer] and
 * abundances[nlayer][nspecies] as read from the atmosphere file (bottom -> top).  imol: species
 * indices of the fitted molecules; imetals: every species but H2, He, H-, e-.  Parameter vector
 * layout (BARTfunc.py:176-181): [PT (npt) | radius (nrad) | cloud top (ncloud) | scattering
 * (one slot unless nray is 0: 1 Lecavelier log-extinction; 2 polar, whose slot's value is unused as
 * in BARTfunc) | log10 abundance factors (nmolfit)].                                            */
int  bart_converter_init(int pt_type, int npt, const double *pt_args, int tint_thorngren,
                         const double *pressure_bar, const double *abundances, int nmolfit,
                         const int *imol, int nmetals, const int *imetals, int iH2, int iHe,
                         double tmin, double tmax, int nrad, int ncloud, int nray);
int  bart_converter_npars(void);

/* replaces code/BARTfunc.py:320-360 for a batch: params[nmodels][npars] -> profiles in
 * run_transit's layout (host buffers; parity/debug use).  status: 0, BART_REJ_TBOUNDS or
 * BART_REJ_ABUND.  knobs_out (may be NULL) [3][nmodels]: radius, cloud top, scattering.          */
int  bart_profiles_from_params(const double *params, int nmodels, int npars, double *profiles,
                               int n_in, int *status, double *knobs_out);

/* replaces one BARTfunc.py worker iteration (309-399) for a batch of proposals:
 * parameters -> band fluxes; profiles and spectra never leave the device.  Rejected proposals
 * get -1 in every band.                                                                         */
int  bart_bandflux_from_params(const double *params, int nmodels, int npars, double *bandflux,
                               int *status);
int  bart_bandflux_from_params_device(const double *d_params, int nmodels, int npars,
                                      double *d_bandflux, int *d_status);

/* contiguous block of chains owned by `rank` (sizes differ by at most one)                      */
void bart_chain_block(int nchains, int world, int rank, int *lo, int *hi);

/* replaces MCcubed.mc.mcmc for walk='demc' (mcmc.py:196-345 set-up and initial chi-squared,
 * 518-625 generation loop; chi-squared and priors of src_c/chisq.c:111-142,
 * src_c/include/stats.h:72-103; MC3 passes priorlow for both prior widths).  params[nchains][npars]
 * are the chains' starting points; stepsize > 0 free, 0 fixed, < 0 shared with parameter
 * -stepsize (1-based).  ndata must equal the number of filters.  With a communicator
 * (bart_comm_init) every rank evaluates its block of chains and one all-gather per generation
 * shares the band fluxes; the proposal and Metropolis steps run redundantly on every rank.
 * Same as bart_mcmc_init_ensemble with nretr = 1.                                               */
int  bart_mcmc_init(int nchains, int npars, const double *params, const double *pmin,
                    const double *pmax, const double *stepsize, const double *prior,
                    const double *priorlow, int ndata, const double *data, const double *uncert,
                    double fgamma, double fepsilon, int burnin);
/* An ensemble of nretr >= 1 independent retrievals of the same planet in one loop: each has its
 * own starting points params[nretr][nchains][npars], data and uncert[nretr][ndata]; the forward
 * model, filters, converter, bounds, step sizes, priors, fgamma, fepsilon and burnin are shared.
 * Every generation evaluates the nretr x nchains models (model g = r * nchains + c) as one batch
 * (split over the ranks like the chains of one retrieval); proposals, Metropolis steps, best fits
 * and snooker histories stay within each retrieval, so retrieval r comes out bit-identical to the
 * same retrieval run alone.  After it, every call below takes and returns its arrays behind a
 * leading [nretr] axis, each retrieval's slice shaped as documented for one retrieval.           */
int  bart_mcmc_init_ensemble(int nretr, int nchains, int npars, const double *params,
                             const double *pmin, const double *pmax, const double *stepsize,
                             const double *prior, const double *priorlow, int ndata,
                             const double *data, const double *uncert, double fgamma,
                             double fepsilon, int burnin);
/* retrievals of the current loop: 1 after bart_mcmc_init, 0 before any init                     */
int  bart_mcmc_nretr(void);
/* MC3's `resume` (mcmc.py:254-269) for walk='demc': call bart_mcmc_init with the chains' last
 * states of the previous run (oldparams[:, :, -1] in the free columns), then this with nold = the
 * previous run's iterations per chain (they count towards burn-in, mcmc.py:616) and curmodel
 * [nretr][nchains][ndata] = the last column of the previous run's `savemodel` array (a chain whose
 * proposals are rejected keeps showing it, mcmc.py:649-651; NULL: zeros, as without savemodel).
 * nold is shared by the retrievals.  Before the first bart_mcmc_run.  (The reference's snooker
 * resume rebuilds its history from the log file's text and is not offered.)                     */
int  bart_mcmc_resume(int nold, const double *curmodel);
/* niter generations without a host round trip.  The random streams are the caller's, in MC3's
 * shapes with chainsize = niter (mcmc.py:484-507) behind the retrieval axis:
 * support[nretr][niter][nchains][nfree], r1/r2[nretr][nchains][niter] (chain indices within the
 * retrieval), unif/ugamma[nretr][niter][nchains].  An out-of-range r1/r2 is refused with the
 * retrieval, generation and chain named.                                                          */
int  bart_mcmc_run(int niter, const double *support, const int *r1, const int *r2,
                   const double *unif, const double *ugamma);
/* replaces MCcubed.mc.mcmc for walk='snooker' -- the walk every BART example configures
 * (examples/WASP-12b/BART.cfg:118) -- DE-MC with snooker updates drawn from the sample history Z
 * (ter Braak & Vrugt 2008): Z set-up and evaluation of the hsize*nchains initial samples
 * (mcmc.py:357-470), proposals (527-561), Metropolis factor of projected jumps (603-609), Z
 * update every `thinning` generations (653-660).  Call after bart_mcmc_init.
 * z0[nretr][hsize][nchains][nfree]: initial samples of the free parameters (the reference draws
 * them uniformly in [pmin, pmax]); hsize > nchains as mcmc.py:233-235 enforces is the caller's
 * job.  hsize and thinning are shared: every retrieval's history grows on the same schedule.     */
int  bart_mcmc_snooker_init(int hsize, int thinning, const double *z0);
/* niter snooker generations without a host round trip.  Random streams in the order mcmc.py
 * consumes them, behind the retrieval axis: support[nretr][niter][nchains][nfree],
 * unif/ugamma[nretr][niter][nchains] (490-497); per generation i1, i2 (flat indices into the
 * retrieval's own history, its first Zsize-1 rows x nchains), iz (row), ic (chain), each
 * [nretr][niter][nchains] (529-539); usnooker[rows][nfree]: the uniform(1.2, 2.2) factors of the
 * chains with ugamma < 0.1 in the reference's draw order (545-556), all retrievals' rows one
 * retrieval after the other; usn_offset[nretr][niter+1] their absolute first rows, generation i
 * of retrieval r owning rows usn_offset[r][i] .. usn_offset[r][i+1] (so usn_offset[r][0] ==
 * usn_offset[r-1][niter] and rows = usn_offset[nretr-1][niter]).                                 */
int  bart_mcmc_run_snooker(int niter, const double *support, const int *i1, const int *i2,
                           const int *iz, const int *ic, const double *usnooker,
                           const int *usn_offset, const double *unif, const double *ugamma);
/* Seeded runs: random streams drawn on the device instead of passed in.  bart_mcmc_seed, after
 * bart_mcmc_init(_ensemble), sets keys[nretr][2], one 128-bit Philox4x64-10 key per retrieval.
 * bart_mcmc_run_seeded(niter) then runs niter generations of the initialised walk (DE-MC, or
 * snooker after bart_mcmc_snooker_init) with MC3's proposal constructions fed by draws that are
 * pure functions of (key, purpose, global iteration, chain, element) -- the counter layout is in
 * bart_b200/csrc/philox.cuh -- so retrieval r of an ensemble equals a lone run with r's key, and
 * host-stream and seeded calls may alternate.  A seeded chain is not MC3's chain (the random
 * numbers differ); it is replayed exactly by bart_mcmc_run* fed the streams bart_mcmc_get returns.
 * bart_mcmc_run_seeded refuses to run before bart_mcmc_seed.                                     */
int  bart_mcmc_seed(const unsigned long long *keys);
int  bart_mcmc_run_seeded(int niter);
/* Keep retrievals keep[0] < keep[1] < ... < keep[nkeep-1] (positions in the current loop) and
 * drop the others: afterwards the loop has nkeep retrievals, retrieval j being the old keep[j], and
 * every call takes and returns arrays behind the new [nkeep] axis.  This is how an ensemble stops
 * each retrieval at its own convergence: the retrievals that are done leave, and the next run
 * calls evaluate only the others' models.  One gather launch moves the kept retrievals' state
 * (chains, best fits, data, Philox keys, snooker histories) into buffers sized for nkeep; the
 * dropped retrievals' device memory is freed.  A kept retrieval's chains are unchanged: it goes on
 * exactly as it would have in the larger loop, seeded calls included (draws depend on the global
 * iteration, which retaining does not touch).  bart_mcmc_get returns the kept retrievals' state;
 * what describes the last run call ("allparams", "allmodel", "models", the streams) is refused
 * until the next run call, so fetch it before retaining.  Allowed any time after
 * bart_mcmc_init_ensemble, before the first run and before bart_mcmc_snooker_init too; keeping
 * every retrieval is a no-op.  Refused: nkeep < 1 or > nretr, positions out of range, not strictly
 * increasing, or repeated.                                                                      */
int  bart_mcmc_retain(int nkeep, const int *keep);
/* "allparams" [nchains][nfree][niter] (MC3's `savefile` array, BART's output.npy), "allmodel"
 * [nchains][ndata][niter] (MC3's `savemodel` array, mcmc.py:636-651,849-850: the model of every
 * chain's current state, zeros until its first acceptance like the reference), "params",
 * "currchisq", "numaccept", "outbounds", "bestp", "bestchisq", "bestmodel", "models", and for
 * snooker "Z" [Zsize][nchains][npars], "Zchisq" [Zsize][nchains]; each behind a leading [nretr]
 * (bestp [nretr][npars], bestchisq [nretr], bestmodel [nretr][ndata]), retrieval-major; with
 * nretr = 1 the layouts are those of one retrieval.  The last run call's random streams, host or
 * seeded, come back as doubles in the layouts bart_mcmc_run / bart_mcmc_run_snooker take them:
 * "support", "unif", "ugamma", and "r1", "r2" after a DE-MC call or "i1", "i2", "iz", "ic",
 * "usnooker", "usn_offset" after a snooker call.  Returns the number of doubles written or < 0. */
long long bart_mcmc_get(const char *name, double *out, long long capacity);

#ifdef __cplusplus
}
#endif
#endif /* BART_B200_H */
