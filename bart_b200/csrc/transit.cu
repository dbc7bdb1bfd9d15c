// transit.cu -- the C ABI of libbart_b200 (include/bart_b200.h): process-global state, init
// sequence, batched execution, timing, introspection and the multi-GPU exchange.
//
// Mirrors the stage sequence of the reference's transit_init (transit/src/transit.c:25-74) and
// run_transit/do_transit (118-214), but everything per-model runs on the device, batched over
// models, with no per-call allocation, no file output inside the MCMC loop (the reference's
// printflux/printmod rewrite the spectrum file on every call, eclipse.c:355-380,
// slantpath.c:510-555; see DESIGN.md "deviations") and no host round trips between stages.
// Host resources are owned by the types of cuda_host.hpp (buffers, staging) and host.hpp (files):
// a configuration's state is one Config value, released whole by reset_state.
#include "../../include/bart_b200.h"
#include "host.hpp"
#include "cuda_host.hpp"
#include "kernels.hpp"
#include "column_math.cuh"
#include "builder.hpp"
#include "retrieval.hpp"
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <cstdarg>
#include <cstring>
#include <cstdlib>
#include <cmath>
#include <string>
#include <vector>
#include <map>
#include <algorithm>
#include <functional>
#include <optional>
#include <sys/stat.h>

namespace bart {

// ---------------------------------------------------------------------------------------
// errors
struct BartError {};
static int g_error_mode = 0;
static bool g_error_pending = false;
static char g_error_msg[4096] = "";
int g_verb = 2;

void fail(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error_msg, sizeof(g_error_msg), fmt, ap);
  va_end(ap);
  g_error_pending = true;
  if (g_error_mode == 0) {
    // reference behaviour: message, then exit(EXIT_FAILURE) (transit.h:91-98)
    fprintf(stderr, "\nTransit ERROR :: %s\n", g_error_msg);
    exit(EXIT_FAILURE);
  }
  throw BartError();
}

void warn(int level, const char *fmt, ...) {
  if (g_verb < level) return;
  va_list ap;
  va_start(ap, fmt);
  fprintf(stderr, "Transit WARNING :: ");
  vfprintf(stderr, fmt, ap);
  fprintf(stderr, "\n");
  va_end(ap);
}

static void info(int level, const char *fmt, ...) {
  if (g_verb < level) return;
  va_list ap;
  va_start(ap, fmt);
  vfprintf(stdout, fmt, ap);
  va_end(ap);
}

// ---------------------------------------------------------------------------------------
// profiling: per-kernel CUDA-event timing on the library stream
struct KStat { long long launches = 0; double ms = 0; };
struct PendingEv { std::string name; cudaEvent_t a, b; };

// Everything one transit_init configuration owns; free_memory and the next transit_init drop it
// whole (reset_state).
struct Config {
  bool init = false;
  Options opt;
  Atmosphere atm;
  Molecules mol;
  Tli tli;
  OpacityGrid og;
  std::vector<CiaTable> cia;
  std::vector<double> wn;
  std::vector<double> angles;
  DevConfig dc{};
  Knobs knobs{};
  // static device arrays
  DevBuf<double> d_grid, d_gtemp, d_wn, d_press, d_mass, d_pol;
  DevBuf<double> d_ciaPQ[kMaxCia], d_ciaT[kMaxCia];
  // batch buffers
  DevBuf<double> d_prof, d_tabs, d_spec, d_wts, d_tau, d_band, d_ext, d_flush;
  DevBuf<int> d_status, d_status_col, d_last;
  PinnedBuf<int> h_status;                 // pinned staging for per-model status
  PinnedBuf<double> h_lean;                // pinned staging of the small-call path (bart_run_batch)
  DevBuf<double> d_kr0, d_kcloud, d_klogext;
  DevBuf<int> d_kflag;
  int knob_models = 0;
  // filters
  int nfilters = 0;
  DevBuf<int> d_fstart, d_fcount, d_foffset;
  DevBuf<double> d_fweight, d_fstar;
  bool have_star = false;
  double rprs2 = 1.0;
  // energy-balance rejection (BARTfunc.py:366-383), applied wherever band fluxes are produced
  bool eb_on = false;
  double eb_ein = 0.0, eb_scale = 0.0;
  int last_batch = 0;
  BuilderPtr builder;
  // line-by-line forward mode (no opacity file)
  bool lbl = false;
  DevBuf<double> d_lbl_ext, d_lbl_dens;
  std::vector<double> h_lbl_T;
  std::vector<int> h_lbl_status;
  // input converter (retrieval.hpp)
  ConvConfig conv{};
  DevBuf<double> d_cpress, d_cbase, d_cratio, d_cparams, d_csmooth, d_cnodex;
  DevBuf<int> d_cnodeseg;
  DevBuf<int> d_cstatus;
  const int *pre_status = nullptr;         // converter rejections of the batch being launched
  // DE-MC loop: `mc` holds views of these
  McmcDev mc{};
  bool mc_ready = false;
  int mc_lo = 0, mc_hi = 0, mc_pad = 0;
  struct {
    DevBuf<double> pmin, pmax, prior, priorlow, data, uncert, params, nextp, currchisq, nextchisq, c2,
        bestp, bestchisq, bestmodel, numaccept, support, unif, ugamma, allparams, zbest;
    DevBuf<int> outbounds, outflag, iter, r1, r2, zsize, noproj, slot;
  } mcb;
  DevBuf<double> d_mcband, d_mcgather, d_mccur, d_mcallm;
  cudaGraphExec_t mc_graph = nullptr;      // destroyed by reset_state
  // snooker walk: sample history Z
  DevBuf<double> d_Z, d_Zchisq, d_snk_usn;
  DevBuf<int> d_snk_idx, d_snk_off;
  int mc_zsize = 0;                        // host mirror of the device row counter
  size_t mc_zcap = 0;                      // rows allocated
  std::vector<double> mc_ztemplate;        // [nretr][nchains][npars] what an unfilled row holds
};

// The process: the device, its streams, the communicator and peer window, profiling and debug
// switches outlive configurations.
struct State : Config {
  int device = -1;
  cudaStream_t stream = nullptr;          // compute (and default copy) stream
  cudaStream_t s_h2d = nullptr, s_d2h = nullptr;   // copy streams of the pipelined host path
  std::vector<cudaEvent_t> ev_pool;                // its events (created once)
  // debug
  bool keep = false;
  int use_tma = 1;
  // profiling
  bool profile = false;
  std::map<std::string, KStat> stats;
  std::vector<PendingEv> pending;
  long long launches = 0;
  cudaEvent_t t0 = nullptr, t1 = nullptr;
  // comm
  void *nccl_lib = nullptr;
  void *nccl_comm = nullptr;
  int rank = 0, world = 1;
  // peer window of the fused band-integration + all-gather (kernels.hpp PeerOut)
  bool p2p = false;
  char *pw_base = nullptr;                 // local allocation: window | flags | gen | done | err
  void *pw_peer[kMaxPeers] = {};           // peers' allocations mapped through CUDA IPC
  long long pw_cap = 0;
  PeerOut pw{};
  unsigned long long *pw_gen = nullptr, *pw_flags = nullptr;
  int *pw_err = nullptr;
};
// Never destroyed: a destructor would run at exit() (error mode 0, or the normal end of the
// process) and call cudaFree while the CUDA runtime is being torn down.  The process's device
// memory goes with the process.
static State &G = *new State;

struct KernelScope {
  const char *name;
  cudaEvent_t a = nullptr, b = nullptr;
  explicit KernelScope(const char *n) : name(n) {
    G.launches++;
    if (G.profile) {
      cudaEventCreate(&a); cudaEventCreate(&b);
      cudaEventRecord(a, G.stream);
    }
  }
  ~KernelScope() {
    if (G.profile) {
      cudaEventRecord(b, G.stream);
      G.pending.push_back({name, a, b});
    }
  }
};

static void drain_profile() {
  for (auto &p : G.pending) {
    cudaEventSynchronize(p.b);
    float ms = 0;
    cudaEventElapsedTime(&ms, p.a, p.b);
    KStat &k = G.stats[p.name];
    k.launches++; k.ms += ms;
    cudaEventDestroy(p.a); cudaEventDestroy(p.b);
  }
  G.pending.clear();
}

static void check_launch(const char *what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) fail("kernel launch '%s' failed: %s", what, cudaGetErrorString(e));
}

// a layer count the column kernels cannot run (column_smem_fits): refused by transit_init
static void fail_layer_limit() {
  const DevConfig &c = G.dc;
  fail("%s geometry supports at most %d layers with %d line-list molecule(s) and %d CIA table(s) "
       "(%d given): the column kernels stage a model's table whole in the shared memory of one block",
       c.eclipse ? "eclipse" : "transit", column_layer_limit(c), c.ngmol, c.ncia, c.nlayer);
}

// ---------------------------------------------------------------------------------------
// device
static void ensure_device() {
  if (G.stream) return;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    fail("no CUDA device available (%s): libbart_b200 has no CPU path",
         e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
  if (G.device < 0) {
    const char *s = getenv("BART_DEVICE");
    if (!s) s = getenv("LOCAL_RANK");
    G.device = s ? atoi(s) % n : 0;
  }
  if (G.device >= n) fail("device ordinal %d out of range (%d devices)", G.device, n);
  CUDA_OK(cudaSetDevice(G.device));
  cudaDeviceProp p;
  CUDA_OK(cudaGetDeviceProperties(&p, G.device));
  if (p.major < 10)
    fail("device %d (%s, sm_%d%d) is not a Blackwell sm_100 part; this library ships sm_100a "
         "code only", G.device, p.name, p.major, p.minor);
  CUDA_OK(cudaStreamCreateWithFlags(&G.stream, cudaStreamNonBlocking));
  CUDA_OK(cudaStreamCreateWithFlags(&G.s_h2d, cudaStreamNonBlocking));
  CUDA_OK(cudaStreamCreateWithFlags(&G.s_d2h, cudaStreamNonBlocking));
  CUDA_OK(cudaEventCreate(&G.t0));
  CUDA_OK(cudaEventCreate(&G.t1));
  const char *t = getenv("BART_NO_TMA");
  G.use_tma = (t && atoi(t)) ? 0 : 1;
}

// n elements of src -> b (at least one element), queued on the library stream
template <class T> static const T *upload_queued(DevBuf<T> &b, const T *src, size_t n) {
  b.ensure(std::max<size_t>(n, 1));
  if (n) CUDA_OK(cudaMemcpyAsync(b.p, src, n * sizeof(T), cudaMemcpyHostToDevice, G.stream));
  return b.p;
}

// ---------------------------------------------------------------------------------------
// init pieces
static void setup_sampling() {
  Options &o = G.opt;
  double lo, hi;
  // makewnsample, makesample.c:308-400
  if (o.wnlow > 0) {
    if (o.wnfct <= 0) fail("User specified wavenumber factor is negative (%g).", o.wnfct);
    lo = o.wnlow * o.wnfct;
  } else if (o.wlhigh > 0) {
    if (o.wlfct <= 0) fail("User specified wavelength factor is negative (%g).", o.wlfct);
    lo = 1.0 / (o.wlhigh * o.wlfct);
  } else fail("Initial wavenumber (nor final wavelength) were correctly provided by the user.");
  if (o.wnhigh > 0) {
    if (o.wnfct < 0) fail("User specified wavenumber factor is negative (%g).", o.wnfct);
    hi = o.wnhigh * o.wnfct;
  } else if (o.wllow > 0) {
    if (o.wlfct < 0) fail("User specified wavelength factor is negative (%g).", o.wlfct);
    hi = 1.0 / (o.wllow * o.wlfct);
  } else fail("Final wavenumber (nor initial wavelength) were correctly provided by the user.");
  if (o.wndelt <= 0) fail("Incorrect wavenumber spacing (%g), it must be positive.", o.wndelt);
  G.wn = make_sampling(lo, hi, o.wndelt, 1);
}

// CIA tables pre-folded through the wavenumber spline.  The reference interpolates, per model and
// per layer, (1) every table row in temperature and (2) the resulting column in wavenumber
// (bicubicinterpolate, crosssec.c:353-428).  Both steps are linear in the table values and step
// (2) does not depend on the model, so it is applied ONCE here to the table columns P_k = y(:,T_k)
// and to their temperature second derivatives Q_k = z(:,T_k); a model then needs only the four
// cubic coefficients of step (1) per layer.
static void setup_cia() {
  const int nw = (int)G.wn.size();
  G.dc.ncia = (int)G.cia.size();
  if (G.dc.ncia > kMaxCia) fail("at most %d cross-section files are supported (%d given)", kMaxCia, G.dc.ncia);
  for (int f = 0; f < G.dc.ncia; f++) {
    const CiaTable &c = G.cia[f];
    const int nx = (int)c.wn.size(), nt = (int)c.temp.size();
    if (c.wn[0] > G.wn[0] || c.wn[nx - 1] < G.wn[nw - 1])
      fail("The wavelength range [%.2f, %.2f] cm-1 of the cross-section file:\n  '%s',\ndoes not "
           "cover Transit's wavelength range [%.2f, %.2f] cm-1.", c.wn[0], c.wn[nx - 1],
           c.file.c_str(), G.wn[0], G.wn[nw - 1]);
    std::vector<double> P, Q;
    fold_cia_table(c, G.wn, P, Q);
    std::vector<double> PQ = pack_cia_quads(P, Q, nt, nw, kEclPad);   // [T_k][wave][4] + padding
    upload(G.d_ciaPQ[f], PQ); upload(G.d_ciaT[f], c.temp);
    G.dc.ciaPQ[f] = G.d_ciaPQ[f].p; G.dc.ciaT[f] = G.d_ciaT[f].p;
    G.dc.cia_nt[f] = nt;
    G.dc.cia_nspec[f] = (int)c.species.size();
    for (size_t s = 0; s < c.species.size(); s++) {
      int idx = -1;
      for (int j = 0; j < G.atm.nspec(); j++) if (G.atm.species[j] == c.species[s]) idx = j;
      if (idx < 0)
        fail("Cross-section species '%s' from file '%s' does not match any in the atmsopheric "
             "file.", c.species[s].c_str(), c.file.c_str());
      G.dc.cia_spec[f][s] = idx;
    }
  }
}

static void load_grid_to_device(const std::string &path) {
  OpacityGrid &g = G.og;
  if (g.nlayer != G.atm.nlayer())
    fail("Opacity grid has %ld layers but the atmosphere has %d.", g.nlayer, G.atm.nlayer());
  if (g.nwave != (long)G.wn.size())
    fail("Opacity grid has %ld wavenumber samples but the configuration asks for %zu.", g.nwave, G.wn.size());
  // device layout: [layer][temp][wave][gms], molecule axis innermost (device.cuh)
  const int gms = g.nmol == 1 ? 1 : (int)((g.nmol + 1) / 2 * 2);
  G.dc.gms = gms;
  const size_t ncell = (size_t)g.nlayer * g.ntemp;
  const size_t cell_in = (size_t)g.nmol * g.nwave, cell_out = (size_t)gms * g.nwave;
  G.d_grid.ensure(ncell * cell_out + (size_t)kEclPad * gms);   // + padding (kernels.hpp kEclPad)
  CUDA_OK(cudaMemsetAsync(G.d_grid.p + ncell * cell_out, 0, (size_t)kEclPad * gms * sizeof(double), G.stream));
  const Fd fd(path.c_str(), O_RDONLY);
  if (fd < 0) fail("Opening opacity file '%s' failed.", path.c_str());
  long long fpos = g.data_offset;
  // stream whole (layer, temperature) cells through the pinned staging (files reach tens of GB at
  // high resolution); each chunk is re-laid out on the device while the next is read
  const size_t cells_per_chunk = std::max<size_t>(1, PinnedStage::kBytes / (cell_in * 8));
  DevBuf<double> d_stage[2] = {DevBuf<double>(cells_per_chunk * cell_in), DevBuf<double>(cells_per_chunk * cell_in)};
  PinnedStage st(cells_per_chunk * cell_in * 8);
  for (size_t cell = 0; cell < ncell;) {
    const size_t nc = std::min(cells_per_chunk, ncell - cell);
    const size_t want = nc * cell_in * 8;
    double *d_in = d_stage[st.next()].p;
    if (!st.put(fd, fpos, want, d_in, G.stream, [&] {
          launch_grid_relayout(d_in, G.d_grid.p + cell * cell_out, (int)nc, (int)g.nmol, gms, (int)g.nwave,
                               G.stream);
        }))
      fail("Opacity file '%s' is truncated.", path.c_str());
    fpos += (long long)want;
    cell += nc;
  }
  cudaStreamSynchronize(G.stream);
  check_launch("grid_relayout");
}

static void finish_grid_config() {
  OpacityGrid &g = G.og;
  if (g.nmol > kMaxGridMol) fail("at most %d line-list molecules are supported", kMaxGridMol);
  G.dc.ntemp = (int)g.ntemp; G.dc.ngmol = (int)g.nmol;
  upload(G.d_gtemp, g.temp);
  G.dc.gtemp = G.d_gtemp.p;
  G.dc.grid = G.d_grid.p;
  for (int m = 0; m < g.nmol; m++) {
    int idx = -1;
    for (int j = 0; j < G.atm.nspec(); j++) if (G.mol.id[j] == g.molid[m]) idx = j;   // valueinarray, extinction.c:575
    if (idx < 0) fail("Opacity-grid molecule ID %d is not among the atmospheric species.", g.molid[m]);
    G.dc.gmol_spec[m] = idx;
  }
}

static void reset_state() {
  if (G.mc_graph) cudaGraphExecDestroy(G.mc_graph);
  static_cast<Config &>(G) = Config();
}

static void do_init(int argc, char **argv) {
  if (G.init) reset_state();
  G.opt = Options();
  parse_options(argc, argv, G.opt);
  Options &o = G.opt;
  // acceptgenhints, argum.c:773-911
  if (o.solution != "eclipse" && o.solution != "transit")
    fail("Solution kind '%s' is invalid.\nCurrently Accepted are:\n transit\n eclipse", o.solution.c_str());
  if (o.nwidth < 1) fail("Times of maximum width has to be greater than one: %g", (double)o.nwidth);
  if (o.ethreshold <= 0) fail("Extinction-coefficient threshold (%.3e) has to be positive.", o.ethreshold);
  if (o.refradius < 0) fail("Reference radius level (%g) must be positive.", o.refradius);
  if (o.refpress < 0) fail("Reference pressure level (%g) must be positive.", o.refpress);
  if (o.gsurf < 0) fail("Surface gravity (%g cm s^-2) must be positive.", o.gsurf);
  if (o.raddelt != -1) fail("raddelt %g: resampling the atmosphere to an equidistant radius grid is "
                            "not supported (BART always uses the atmosphere-file layers)", o.raddelt);
  if (o.taulevel != 1) fail("slantpath:: totaltau:: Level %i of detail has not been implemented to "
                            "compute optical depth.", o.taulevel);
  if (o.modlevel != 1 && o.modlevel != -1)          // slantpath.c:497-503
    fail("slantpath:: modulationperwn:: Level %i of detail has not been implemented to compute "
         "modulation.", o.modlevel);
  ensure_device();

  info(2, "--------------------------------------------------\n"
          "        TRANSIT (bart_b200, sm_100a)\n"
          "--------------------------------------------------\n");
  setup_sampling();
  read_atmosphere(o.atm, G.atm);
  // BART's atmosphere files carry number abundances ('q number', TEA / makeatm.py) and BARTfunc does
  // its own abundance scaling: the reference's mass-abundance branch (readatm.c:122-159,
  // transit.h:58-69 with at->mass) and its qmol/qscale hints are not built -- refuse them rather
  // than compute densities from the wrong kind of abundance
  if (G.atm.mass_abund)
    fail("Atmosphere file '%s' gives abundances by mass ('q mass'); only number abundances "
         "('q number') are supported.", o.atm.c_str());
  if (!o.qmol.empty() || !o.qscale.empty())
    fail("The 'qmol' / 'qscale' abundance-scaling options are not supported (scale the abundances "
         "in the run_transit input, as BARTfunc.py does).");
  read_molecules(o.molfile, G.atm, G.mol);
  read_tli_header(o.linedb, G.tli);
  const int nl = G.atm.nlayer(), ns = G.atm.nspec(), nw = (int)G.wn.size();
  if (ns > kMaxSpec) fail("at most %d atmospheric species are supported", kMaxSpec);
  // makeradsample's temperature check against the TLI range (makesample.c:488-503)
  for (int i = 0; i < nl; i++) {
    if (G.atm.temp[i] * G.atm.tfct < G.tli.tmin)
      fail("The layer %d in the atmospheric model has a lower temperature (%.1f K) than the lowest "
           "allowed TLI temperature (%.1f K).", i, G.atm.temp[i], G.tli.tmin);
    if (G.atm.temp[i] * G.atm.tfct > G.tli.tmax)
      fail("The layer %d in the atmospheric model has a higher temperature (%.1f K) than the "
           "highest allowed TLI temperature (%.1f K).", i, G.atm.temp[i], G.tli.tmax);
  }

  DevConfig &c = G.dc;
  c = DevConfig();
  c.nlayer = nl; c.nspec = ns; c.nwave = nw;
  c.eclipse = o.solution == "eclipse";
  c.transparent = o.transparent ? 1 : 0;
  c.modlevel = o.modlevel;
  c.pfct = G.atm.pfct; c.rfct = G.atm.rfct; c.gsurf = o.gsurf; c.p0 = o.refpress;
  c.toomuch = o.toomuch;
  upload(G.d_wn, G.wn); c.wn = G.d_wn.p;
  upload(G.d_press, G.atm.press); c.press = G.d_press.p;
  c.ref_layer = ref_layer_of(G.atm.press.data(), nl, c.p0);
  upload(G.d_mass, G.mol.mass); c.mass = G.d_mass.p;
  upload(G.d_pol, G.mol.pol); c.pol = G.d_pol.p;
  // ray grid (acceptgenhints 878-881; flux(), eclipse.c:262-279)
  G.angles.clear();
  if (c.eclipse) {
    char *dup = strdup(o.raygrid.c_str());
    for (char *t = strtok(dup, " \t"); t; t = strtok(nullptr, " \t")) G.angles.push_back(atof(t));
    free(dup);
    if (G.angles.empty() || (int)G.angles.size() > kMaxAng)
      fail("raygrid must hold between 1 and %d angles", kMaxAng);
    c.nang = (int)G.angles.size();
    std::vector<double> area(c.nang + 1);
    area[0] = 0.0 * kDEG; area[c.nang] = 90.0 * kDEG;
    for (int a = 1; a < c.nang; a++) area[a] = (G.angles[a - 1] + G.angles[a]) * kDEG / 2.0;
    for (int a = 0; a < c.nang; a++) {
      c.inv_mu[a] = 1.0 / cos(G.angles[a] * kDEG);
      c.wgt[a] = pow(sin(area[a + 1]), 2.0) - pow(sin(area[a]), 2.0);
    }
    fill_angle_consts(c);
    // Planck chaining between the columns of one thread (device.cuh): needs the uniform grid that
    // makewnsample always produces (makesample.c:97-104)
    c.planck_cols = 0;
    if (nw > kEclThreads) {
      const double dwn = (G.wn[nw - 1] - G.wn[0]) / (nw - 1);
      double dev = 0.0;
      for (int i = 1; i < nw; i++) dev = std::max(dev, fabs((G.wn[i] - G.wn[i - 1]) - dwn));
      if (dev > 1e-9 * dwn) fail("internal: the wavenumber grid is not uniform (max deviation %g)", dev);
      c.planck_cols = kEclThreads;
      c.planck_step = cH * cLS / cKB * kEclThreads * dwn;
    }
  }
  upload_exp_table(c, G.stream);
  const double srad = o.starrad * kSUNRADIUS;                      // geometry.c:36,50
  c.inv_srad2 = 1.0 / (srad * srad);

  // knobs: process-wide defaults from the configuration
  Knobs &k = G.knobs;
  k = Knobs();
  k.r0_all = o.refradius;
  k.cloud_flag_all = o.cloud_flag; k.cloudext_all = o.cloudext;
  k.cloudtop_all = o.cloudtop; k.cloudbot_all = o.cloudbot;
  k.scat_flag_all = o.scat_flag; k.scat_logext_all = o.scat_logext;

  // opacity(): opacity.c:8-214
  bool have_file = false;
  if (!o.opacityfile.empty()) {
    struct stat st;
    have_file = stat(o.opacityfile.c_str(), &st) == 0 && S_ISREG(st.st_mode);
  }
  G.lbl = false;
  if (o.opacityfile.empty()) {
    // opacity.c:28-36: no opacity file -> Voigt profiles only; tau() computes every layer line by
    // line at the layer's own temperature (tau.c:163-175,253-264)
    if (!G.tli.present) fail("Neither an opacity file nor a TLI line list (linedb) was given.");
    if (o.justOpacity) fail("--justOpacity needs 'opacityfile'.");
    info(2, "No opacity file: line-by-line extinction at every run_transit call.\n");
    G.lbl = true;
    builder_lbl_cells(G.builder, G.opt, G.atm, G.mol, G.tli, G.wn, G.stream, 0, nullptr, nullptr,
                      nullptr, nullptr);               // Voigt table + line list on the device
    c.lbl = 1; c.ntemp = 2; c.ngmol = 1; c.gms = 1;
    upload(G.d_gtemp, std::vector<double>{G.tli.tmin, G.tli.tmax});
    c.gtemp = G.d_gtemp.p;
    c.gmol_spec[0] = 0;
  } else {
  // a temperature-sliced build ($BART_TSLICE, one process per GPU) writes into the file the other
  // slices are creating: its existence does not mean it is complete
  const bool sliced = o.justOpacity && getenv("BART_TSLICE") != nullptr;
  if (!have_file || sliced) {
    if (!G.tli.present) fail("Cannot build the opacity grid '%s': no TLI line list (linedb) given.", o.opacityfile.c_str());
    info(2, "Calculating new grid of opacities: '%s'.\n", o.opacityfile.c_str());
    builder_run_and_write(G.builder, G.opt, G.atm, G.mol, G.tli, G.wn, G.stream, o.opacityfile);
  }
  if (o.justOpacity) {            // transit.c:133-136 opabreak: nothing else to do
    G.init = true;
    return;
  }
  if (!read_opacity_header(o.opacityfile, G.og)) fail("Opening opacity file failed.");
  load_grid_to_device(o.opacityfile);
  finish_grid_config();
  }

  // Models with a layer outside the grid's temperature range (line by line: the TLI range) are
  // rejected before the column kernels run, so the Planck exponents x = hc wn/(k T) they can meet
  // lie in [hc wn_min/(k Tmax), hc wn_max/(k Tmin)].  The specialised eclipse kernels evaluate
  // e^x - 1 to degree 4 without a clamp: fine for 0.1 <= x <= 690 (relative error of e^x - 1 below
  // 2.6e-12 e^x/(e^x - 1) <= 2.8e-11); anything wider takes the generic kernel.
  {
    const double tmin = G.lbl ? G.tli.tmin : G.og.temp[0];
    const double tmax = G.lbl ? G.tli.tmax : G.og.temp[G.og.ntemp - 1];
    const double c2 = cH * cLS / cKB;
    c.planck_generic = !(tmin > 0) || c2 * G.wn[nw - 1] / tmin > 690.0 || c2 * G.wn[0] / tmax < 0.1;
  }

  // readcs(): crosssec.c:9-268
  G.cia.resize(o.csfiles.size());
  for (size_t i = 0; i < o.csfiles.size(); i++) read_cia(o.csfiles[i], G.cia[i]);
  setup_cia();

  c.lay.nl = nl; c.lay.ngmol = c.ngmol; c.lay.ncia = c.ncia;
  if (!column_smem_fits(c)) fail_layer_limit();
  G.init = true;
  info(2, "transit_init done: %d layers, %d species, %d wavenumbers, grid %ld T x %ld mol (%.1f MB "
          "in HBM), %d CIA file(s), %s geometry.\n", nl, ns, nw, G.og.ntemp, G.og.nmol,
       (double)bart_grid_bytes() / 1e6, c.ncia, c.eclipse ? "eclipse" : "transit");
}

// ---------------------------------------------------------------------------------------
// batched execution (device-resident inputs)
static Knobs effective_knobs(int nmodels) {
  Knobs k = G.knobs;
  if (G.knob_models != nmodels) { k.r0 = nullptr; k.cloudtop = nullptr; k.scat_flag = nullptr; k.scat_logext = nullptr; }
  return k;
}

// Launch the forward model for models [off, off+count) of a batch of `total` models whose
// buffers (tables, status, keep arrays, per-model knobs) are indexed by the global model number.
static void prepare_batch(int total, int n_in) {
  DevConfig &c = G.dc;
  if (!G.init || G.opt.justOpacity) fail("Transit init not run, please initialize transit.");
  if (n_in < (c.nspec + 1) * c.nlayer)
    fail("run_transit: input has %d values, expected (1+%d species) x %d layers = %d", n_in, c.nspec,
         c.nlayer, (c.nspec + 1) * c.nlayer);
  G.d_tabs.ensure((size_t)total * c.lay.stride());
  G.d_status.ensure(total);
  G.d_status_col.ensure(total);
  if (G.keep) {
    G.d_tau.ensure((size_t)total * c.nwave * c.nlayer);
    G.d_last.ensure((size_t)total * c.nwave);
    CUDA_OK(cudaMemsetAsync(G.d_tau.p, 0, (size_t)total * c.nwave * c.nlayer * sizeof(double), G.stream));
  }
  if (!c.eclipse) G.d_wts.ensure((size_t)total * transit_weights_stride(c.nlayer));
  if (G.lbl) {
    // one extra row: the column kernels also load the (zero-weighted) second bracket plane
    G.d_lbl_ext.ensure(((size_t)total * c.nlayer + 1) * c.nwave + kEclPad);
    G.d_lbl_dens.ensure((size_t)std::max(1, total) * c.nlayer * c.nspec);
    c.grid = G.d_lbl_ext.p;
    c.lbl_dens = G.d_lbl_dens.p;
  }
}

// Line-by-line mode: molecular extinction of models [off, off+count) (those atm_prep accepted)
// into ext[model][layer][wave], by the builder kernels with one plane per (model, layer).
static void lbl_extinction(const double *d_prof, int off, int count, int n_in) {
  DevConfig &c = G.dc;
  const int nl = c.nlayer, nw = c.nwave;
  G.h_lbl_T.resize((size_t)count * nl);
  G.h_lbl_status.resize(count);
  CUDA_OK(cudaMemsetAsync(G.d_lbl_ext.p + (size_t)off * nl * nw, 0,
                          ((size_t)count * nl + 1) * nw * sizeof(double), G.stream));
  CUDA_OK(cudaMemcpy2DAsync(G.h_lbl_T.data(), (size_t)nl * 8, d_prof, (size_t)n_in * 8, (size_t)nl * 8,
                            count, cudaMemcpyDeviceToHost, G.stream));
  CUDA_OK(cudaMemcpyAsync(G.h_lbl_status.data(), G.d_status.p + off, count * sizeof(int),
                          cudaMemcpyDeviceToHost, G.stream));
  CUDA_OK(cudaStreamSynchronize(G.stream));
  std::vector<double> cT;
  std::vector<long long> cout_;
  for (int m0 = 0; m0 < count;) {                       // runs of accepted models
    if (G.h_lbl_status[m0] != 0) { m0++; continue; }
    int m1 = m0;
    while (m1 < count && G.h_lbl_status[m1] == 0) m1++;
    const int ncell = (m1 - m0) * nl;
    cT.resize(ncell); cout_.resize(ncell);
    for (int m = m0; m < m1; m++)
      for (int l = 0; l < nl; l++) {
        cT[(size_t)(m - m0) * nl + l] = G.h_lbl_T[(size_t)m * nl + l] * G.atm.tfct;
        cout_[(size_t)(m - m0) * nl + l] = ((long long)(off + m) * nl + l) * nw;
      }
    KernelScope ks("lbl_extinction");
    builder_lbl_cells(G.builder, G.opt, G.atm, G.mol, G.tli, G.wn, G.stream, ncell, cT.data(),
                      G.d_lbl_dens.p + (size_t)(off + m0) * nl * c.nspec, cout_.data(), G.d_lbl_ext.p);
    G.launches += 5;                                    // kmax, count, scan, fill, widths (+ accumulate)
    m0 = m1;
  }
}

static void launch_models(const double *d_prof, int off, int count, int total, int n_in, double *d_spec) {
  DevConfig &c = G.dc;
  if (count <= 0) return;
  Knobs k = effective_knobs(total);
  if (k.r0) k.r0 += off;
  if (k.cloudtop) k.cloudtop += off;
  if (k.scat_flag) k.scat_flag += off;
  if (k.scat_logext) k.scat_logext += off;
  double *tabs = G.d_tabs.p + (size_t)off * c.lay.stride();
  int *status = G.d_status.p + off;
  double *tau = G.keep ? G.d_tau.p + (size_t)off * c.nwave * c.nlayer : nullptr;
  int *last = G.keep ? G.d_last.p + (size_t)off * c.nwave : nullptr;
  {
    KernelScope ks("atm_prep");
    DevConfig cc = c;
    cc.lbl_model0 = off;
    launch_atm_prep(cc, k, d_prof, n_in, tabs, status, G.pre_status ? G.pre_status + off : nullptr, count, G.stream);
    check_launch("atm_prep");
  }
  if (G.lbl) lbl_extinction(d_prof, off, count, n_in);
  // scattering / cloud terms of the table records (prep_table_row): all zero unless a flag is set
  const bool sc = k.scat_flag || k.cloudtop || k.scat_flag_all != 0 ||
                  (k.cloud_flag_all == 1 && k.cloudext_all != 0.0);
  if (c.eclipse) {
    KernelScope ks("eclipse_column");
    if (!launch_eclipse(c, tabs, status, d_spec, tau, last, count, G.keep, sc, G.use_tma, G.stream)) fail_layer_limit();
    check_launch("eclipse_column");
  } else {
    int *scol = G.d_status_col.p + off;         // cleared by the weights kernel
    double *wts = G.d_wts.p + (size_t)off * transit_weights_stride(c.nlayer);
    {
      KernelScope ks("transit_weights");
      launch_transit_weights(c, tabs, wts, count, G.keep, scol, G.stream);
      check_launch("transit_weights");
    }
    {
      KernelScope ks("transit_column");
      if (!launch_transit(c, tabs, wts, status, scol, d_spec, tau, last, count, G.keep, sc, G.use_tma, G.stream))
        fail_layer_limit();
      check_launch("transit_column");
    }
    launch_merge_status(status, scol, count, G.stream);
    G.launches += 1;                 // merge_status
  }
}

static void run_models_device(const double *d_prof, int nmodels, int n_in, double *d_spec) {
  if (nmodels <= 0) { prepare_batch(0, n_in); return; }
  prepare_batch(nmodels, n_in);
  launch_models(d_prof, 0, nmodels, nmodels, n_in, d_spec);
  G.last_batch = nmodels;
}

static void band_device(const double *d_spec, int nmodels, const int *d_status, double *d_band,
                        bool to_peers = false) {
  if (G.nfilters <= 0) fail("bart_set_filters has not been called");
  if (to_peers && nmodels <= 0) {          // nothing to integrate: still announce this rank
    KernelScope ks("peer_signal");
    launch_peer_signal(G.pw, G.stream);
    check_launch("peer_signal");
    return;
  }
  if (G.eb_on && d_status) {
    KernelScope ks("energy_balance");
    launch_energy_balance(d_spec, G.d_wn.p, G.dc.nwave, G.eb_scale, G.eb_ein, const_cast<int *>(d_status),
                          nmodels, G.stream);
    check_launch("energy_balance");
  }
  KernelScope ks("band_integrate");
  launch_band_integrate(d_spec, G.d_wn.p, G.d_fstart.p, G.d_fcount.p, G.d_foffset.p, G.d_fweight.p,
                        G.have_star ? G.d_fstar.p : nullptr, G.rprs2, d_status, d_band, G.nfilters,
                        G.dc.nwave, nmodels, G.stream, to_peers ? &G.pw : nullptr);
  check_launch("band_integrate");
}

static double peer_timeout_s() {
  const char *e = getenv("BART_PEER_TIMEOUT_S");
  const double v = e ? atof(e) : 120.0;
  return v > 0 ? v : 120.0;
}
// consumer side of the fused all-gather: wait for every rank's block, copy to d_all[rank][count]
static void peer_gather(long long count_per_rank, double *d_all) {
  KernelScope ks("peer_wait_copy");
  launch_peer_wait_copy((const double *)G.pw_base, G.pw_flags, G.pw_gen, G.world, G.pw_cap,
                        count_per_rank, d_all, G.pw_err, G.pw.done + 1,
                        (unsigned long long)(peer_timeout_s() * 1e9), G.stream);
  check_launch("peer_wait_copy");
}

static bool p2p_usable(long long count_per_rank) {
  return G.p2p && G.world > 1 && count_per_rank <= G.pw_cap;
}


// ---------------------------------------------------------------------------------------
// retrieval loop (retrieval.cu): parameters -> band fluxes on the device
static void chain_block(int nchains, int world, int rank, int *lo, int *hi) {
  const int base = nchains / world, extra = nchains % world;
  *lo = rank * base + std::min(rank, extra);
  *hi = *lo + base + (rank < extra ? 1 : 0);
}

// converter + forward model + band integration for `nmodels` parameter vectors on the device.
// No synchronisation: everything is queued on G.stream.
static void ensure_params_buffers(int nmodels) {
  const DevConfig &c = G.dc;
  if (!G.init || G.opt.justOpacity) fail("Transit init not run, please initialize transit.");
  if (!G.conv.ready) fail("bart_converter_init has not been called");
  if (G.nfilters <= 0) fail("bart_set_filters has not been called");
  if (G.lbl) fail("the device-resident retrieval loop needs an opacity grid (set 'opacityfile'); the "
                  "line-by-line mode serves run_transit / bart_run_batch only");
  const int n_in = (c.nspec + 1) * c.nlayer;
  G.d_prof.ensure((size_t)std::max(1, nmodels) * n_in);
  G.d_spec.ensure((size_t)std::max(1, nmodels) * c.nwave);
  G.d_cstatus.ensure(std::max(1, nmodels));
  G.d_kr0.ensure(std::max(1, nmodels)); G.d_kcloud.ensure(std::max(1, nmodels));
  G.d_klogext.ensure(std::max(1, nmodels)); G.d_kflag.ensure(std::max(1, nmodels));
  prepare_batch(nmodels, n_in);
}

static void params_to_bandflux_queued(const double *d_params, int nmodels, int npars, double *d_band,
                                      bool to_peers = false) {
  const DevConfig &c = G.dc;
  const ConvConfig &cc = G.conv;
  if (npars != cc.npars) fail("parameter vectors have %d entries, the converter expects %d", npars, cc.npars);
  if (nmodels <= 0) { if (to_peers) band_device(nullptr, 0, nullptr, d_band, true); return; }
  const int n_in = (c.nspec + 1) * c.nlayer;
  ConvKnobs kn{G.d_kr0.p, G.d_kcloud.p, G.d_klogext.p, G.d_kflag.p};
  {
    KernelScope ks("convert_params");
    launch_convert_params(cc, d_params, npars, G.d_prof.p, n_in, G.d_cstatus.p, kn, nmodels, G.stream);
    check_launch("convert_params");
  }
  // per-model knobs written by the converter (BARTfunc.py:350-360)
  Knobs saved = G.knobs;
  const int saved_models = G.knob_models;
  G.knobs.r0 = cc.nrad ? G.d_kr0.p : nullptr;
  G.knobs.cloudtop = cc.ncloud ? G.d_kcloud.p : nullptr;
  G.knobs.scat_flag = cc.nray ? G.d_kflag.p : nullptr;
  G.knobs.scat_logext = cc.nray ? G.d_klogext.p : nullptr;
  G.knob_models = nmodels;
  G.pre_status = G.d_cstatus.p;
  launch_models(G.d_prof.p, 0, nmodels, nmodels, n_in, G.d_spec.p);
  G.pre_status = nullptr;
  G.knobs = saved;
  G.knob_models = saved_models;
  G.last_batch = nmodels;
  band_device(G.d_spec.p, nmodels, G.d_status.p, d_band, to_peers);
}

static const double *mcmc_evaluate_queued(const double *d_params);

// one DE-MC / snooker generation, queued on G.stream (first: the initial evaluation,
// mcmc.py:310-345)
static void mcmc_generation_queued(int first) {
  McmcDev &mc = G.mc;
  if (!first && mc.walk == 1) {
    KernelScope ks("snooker_propose");
    launch_snooker_propose(mc, G.stream);
    check_launch("snooker_propose");
  } else if (!first) {
    KernelScope ks("demc_propose");
    launch_demc_propose(mc, G.stream);
    check_launch("demc_propose");
  }
  const double *models = mcmc_evaluate_queued(first ? mc.params : mc.nextp);
  const int ntot = mc.nretr * mc.nchains;
  ModelMap mp{G.world, ntot / G.world, ntot % G.world, G.mc_pad};
  {
    KernelScope ks("chisq_accept");
    launch_chisq_accept(mc, models, mp, first, G.stream);
    check_launch("chisq_accept");
  }
}

// band fluxes of one population `d_params` [nretr * nchains][npars] (device): this rank's block of chains
// through the forward model, then the all-gather; returns the buffer chain_model() indexes
static const double *mcmc_evaluate_queued(const double *d_params) {
  McmcDev &mc = G.mc;
  const int nloc = G.mc_hi - G.mc_lo;
  const double *src = d_params + (size_t)G.mc_lo * mc.npars;
  const long long per_rank = (long long)G.mc_pad * mc.ndata;
  const bool fused = p2p_usable(per_rank);
  params_to_bandflux_queued(src, nloc, mc.npars, G.d_mcband.p, fused);
  const double *models = G.d_mcband.p;
  if (fused) {
    // band fluxes went straight into every rank's window from the band-integration kernel
    peer_gather(per_rank, G.d_mcgather.p);
    models = G.d_mcgather.p;
  } else if (G.world > 1) {
    typedef int (*fn_allgather)(const void *, void *, size_t, int, void *, cudaStream_t);
    fn_allgather ag = (fn_allgather)dlsym(G.nccl_lib, "ncclAllGather");
    if (!ag || !G.nccl_comm) fail("multi-rank DE-MC needs bart_comm_init first");
    int rc = ag(G.d_mcband.p, G.d_mcgather.p, (size_t)G.mc_pad * mc.ndata, 8 /*ncclFloat64*/,
                G.nccl_comm, G.stream);
    if (rc != 0) fail("ncclAllGather failed (%d)", rc);
    G.launches++;
    models = G.d_mcgather.p;
  }
  return models;
}

static void finish_stream() {
  cudaError_t e = cudaStreamSynchronize(G.stream);
  if (e != cudaSuccess) fail("CUDA execution failed: %s", cudaGetErrorString(e));
  if (G.profile) drain_profile();
}

// The consumer of the fused all-gather (peer_wait_copy_kernel) gives up on a silent peer after
// $BART_PEER_TIMEOUT_S (default 120 s) and raises this flag instead of hanging; whatever was computed
// from that generation on is garbage, so every path that waited on the window must look at it.
static void check_peer_window(const char *where) {
  if (!G.p2p || G.world <= 1 || !G.pw_err) return;
  int err = 0;
  CUDA_OK(cudaMemcpy(&err, G.pw_err, sizeof(int), cudaMemcpyDeviceToHost));
  if (!err) return;
  CUDA_OK(cudaMemset(G.pw_err, 0, sizeof(int)));
  fail("%s: a rank did not deliver its band fluxes to the peer window within %.0f s (dead or "
       "lagging peer); the results of this call are invalid", where, peer_timeout_s());
}
// all ranks have reached this point (ranks load their grids at different speeds; the first fused
// generation must not start its time-out clock before the slowest one is ready)
static void rank_barrier() {
  if (G.world <= 1 || !G.nccl_comm) return;
  typedef int (*fn_allgather)(const void *, void *, size_t, int, void *, cudaStream_t);
  fn_allgather ag = (fn_allgather)dlsym(G.nccl_lib, "ncclAllGather");
  if (!ag) fail("ncclAllGather not found");
  G.d_mcgather.ensure((size_t)G.world + 1);
  int rc = ag(G.d_mcgather.p + G.world, G.d_mcgather.p, 1, 8 /*ncclFloat64*/, G.nccl_comm, G.stream);
  if (rc != 0) fail("ncclAllGather (barrier) failed (%d)", rc);
  cudaError_t e = cudaStreamSynchronize(G.stream);
  if (e != cudaSuccess) fail("CUDA execution failed: %s", cudaGetErrorString(e));
}

// niter generations of the walk set up in G.mc, queued and awaited
static void mcmc_run_generations(int niter) {
  McmcDev &mc = G.mc;
  CUDA_OK(cudaMemsetAsync(mc.iter, 0, (size_t)mc.nretr * sizeof(int), G.stream));
  if (G.mc_graph) { cudaGraphExecDestroy(G.mc_graph); G.mc_graph = nullptr; }
  ensure_params_buffers(G.mc_hi - G.mc_lo);
  // One generation is a fixed sequence of launches whose only varying input, the iteration
  // number, lives on the device: capture it once and replay it (launch-latency bound at MC3's
  // usual 10-chain populations).  Per-kernel timing and multi-rank runs use plain launches unless
  // BART_MCMC_GRAPH=1.
  const char *genv = getenv("BART_MCMC_GRAPH");
  // (multi-rank: only when the all-gather is the fused peer-window one -- plain kernels, no NCCL node)
  bool use_graph = genv ? atoi(genv) != 0 : (G.world == 1 || p2p_usable((long long)G.mc_pad * mc.ndata));
  if (G.profile || niter < 3) use_graph = false;
  int done = 0;
  if (use_graph) {
    mcmc_generation_queued(0); done = 1;          // warms every lazily configured launch
    const long long before = G.launches;
    cudaGraph_t graph = nullptr;
    CUDA_OK(cudaStreamBeginCapture(G.stream, cudaStreamCaptureModeThreadLocal));
    bool ok = true;
    try { mcmc_generation_queued(0); } catch (BartError &) { ok = false; }
    cudaError_t e = cudaStreamEndCapture(G.stream, &graph);
    const long long per_gen = G.launches - before;
    if (ok && e == cudaSuccess && graph &&
        cudaGraphInstantiate(&G.mc_graph, graph, 0) == cudaSuccess) {
      for (; done < niter; done++) CUDA_OK(cudaGraphLaunch(G.mc_graph, G.stream));
      G.launches += per_gen * (niter - 2);
    } else {
      cudaGetLastError();
      G.launches = before;
      if (!ok) { g_error_pending = false; g_error_msg[0] = 0; }
    }
    if (graph) cudaGraphDestroy(graph);
  }
  for (; done < niter; done++) mcmc_generation_queued(0);
  finish_stream();
  check_peer_window("MCMC generations");
}

}  // namespace bart

using namespace bart;

#define API_BEGIN try {
#define API_END_INT                                   \
  } catch (BartError &) { return -1; }                \
  catch (std::exception & e) {                        \
    snprintf(g_error_msg, sizeof(g_error_msg), "%s", e.what()); g_error_pending = true; return -1; }
#define API_END_VOID                                  \
  } catch (BartError &) { return; }                   \
  catch (std::exception & e) {                        \
    snprintf(g_error_msg, sizeof(g_error_msg), "%s", e.what()); g_error_pending = true; return; }

extern "C" {

// =========================================================================================
// Part 1: the reference boundary
void transit_init(int argc, char **argv) {
  API_BEGIN
  do_init(argc, argv);
  API_END_VOID
}

int get_no_samples(void) { return (int)G.wn.size(); }

void get_waveno_arr(double *waveno_arr, int waveno) {
  const int n = std::min((int)G.wn.size(), waveno);
  if (G.init) for (int i = 0; i < n; i++) waveno_arr[i] = G.wn[i];
  else {
    printf("Transit not initialized, please run init. Values set -1\n");
    for (int i = 0; i < waveno; i++) waveno_arr[i] = -1;
  }
}

void set_radius(double refradius) { G.knobs.r0_all = refradius; }

void set_cloudtop(double cloudtop) {
  G.knobs.cloudtop_all = cloudtop; G.knobs.cloudbot_all = cloudtop + 10;
  G.knobs.cloudext_all = 100; G.knobs.cloud_flag_all = 1;
}

void set_scattering(int flag, double scattering) {
  G.knobs.scat_flag_all = flag; G.knobs.scat_logext_all = scattering;
}

// `savefiles yes` (tau.c:179-190,308-329): the six text dumps of one run_transit call, written to
// the working directory in the reference's layouts (print2dArrayDouble / save1Darray /
// savemolExtion, tau.c:360-518; format %-20.10g).  code/cf.py:68-135 reads tau.dat.
static void write_savefiles(const double *re_input, int n_in) {
  const DevConfig &c = G.dc;
  const int nl = c.nlayer, nw = c.nwave, nf = c.lay.nf();
  std::vector<double> tau((size_t)nw * nl), tab((size_t)c.lay.stride());
  CUDA_OK(cudaMemcpy(tau.data(), G.d_tau.p, tau.size() * 8, cudaMemcpyDeviceToHost));
  CUDA_OK(cudaMemcpy(tab.data(), G.d_tabs.p, tab.size() * 8, cudaMemcpyDeviceToHost));
  std::vector<double> mol((size_t)nl * nw), tot((size_t)nl * nw), cia((size_t)nl * nw);
  if (bart_extinction_batch(re_input, 1, n_in, mol.data(), 0) != 0) return;
  if (bart_extinction_batch(re_input, 1, n_in, tot.data(), 1) != 0) return;
  if (bart_extinction_batch(re_input, 1, n_in, cia.data(), 2) != 0) return;
  const char *fmt = "%-20.10g";
  auto open_dump = [](const char *name, const char *header) {
    File f(name, "w");
    if (!f) fail("cannot open '%s' for writing (savefiles)", name);
    fprintf(f, "\n");
    fputs(header, f);
    return f;
  };
  // per-wavenumber rows [wn][rad], rad[0] = bottom: total, cloud, scattering (save1Darray)
  const File ft = open_dump("total_extion.dat", "# 2D total extinction\n# er [wn][rad]; wn[0]=min(wn), row[0]=bottom (max(p))\n");
  const File fc = open_dump("cloud_extion.dat", "# 2D cloud extinction\n# e_c [wn][rad]; wn[0]=min(wn), row[0]=bottom (max(p))\n");
  const File fs = open_dump("scatt_extion.dat", "# 2D scatt extinction\n# e_s [wn][rad]; wn[0]=min(wn), row[0]=bottom (max(p))\n");
  for (int w = 0; w < nw; w++) {
    const double wn = G.wn[w], wn4 = (wn * wn) * (wn * wn);
    FILE *fl[3] = {ft, fc, fs};
    for (int k = 0; k < 3; k++) {
      fprintf(fl[k], "\nwavenumber: ");
      fprintf(fl[k], fmt, wn);
      fprintf(fl[k], "\n");
      for (int r = 0; r < nl; r++) {
        const double *row = tab.data() + (size_t)(nl - 1 - r) * nf;
        const double v = k == 0 ? tot[(size_t)r * nw + w] : (k == 1 ? row[TabLayout::CLOUD] : row[TabLayout::SCAT] * wn4);
        fprintf(fl[k], fmt, v);
      }
      fprintf(fl[k], "\n");
    }
  }
  // tau.dat [wn][rad], rad[0] = top; CIA.dat [wn][rad], rad[0] = bottom (print2dArrayDouble)
  const File f = open_dump("tau.dat", "# 2D optical depth\n# tau [wn][rad]; wn[0]=min(wn); rad[0]=top (min(p))\n\n");
  const File g = open_dump("CIA.dat", "# 2D CIA extinction\n# e_cs [wn][rad]; wn[0]=min(wn); row[0]=bottom (max(p))\n\n");
  for (int w = 0; w < nw; w++) {
    FILE *fl[2] = {f, g};
    for (int k = 0; k < 2; k++) {
      fprintf(fl[k], "wavenumber: ");
      fprintf(fl[k], fmt, G.wn[w]);
      fprintf(fl[k], "\n");
      for (int r = 0; r < nl; r++) fprintf(fl[k], fmt, k == 0 ? tau[(size_t)w * nl + r] : cia[(size_t)r * nw + w]);
      fprintf(fl[k], "\n\n");
    }
  }
  // mol_extion.dat [rad][wn], rad[0] = bottom (savemolExtion)
  const File m = open_dump("mol_extion.dat", "# mol-line extinction\n# e [rad][wn]; rad[0]=bottom (max(p)); wn[0]=min(wn)\n\n");
  for (int r = 0; r < nl; r++) {
    fprintf(m, "radius: %-20.10g\n", tab[(size_t)(nl - 1 - r) * nf + TabLayout::RAD]);
    for (int w = 0; w < nw; w++) fprintf(m, fmt, mol[(size_t)r * nw + w]);
    fprintf(m, "\n\n");
  }
}

void run_transit(double *re_input, int transint, double *transit_out, int transit_out_size) {
  API_BEGIN
  if (!G.init) { printf("Transit init not run, please initialize transit.\n"); return; }
  int status = 0;
  const int saved = G.knob_models;
  G.knob_models = 0;                         // the single-model call uses the process-wide setters
  const bool saved_keep = G.keep;
  if (G.opt.savefiles) G.keep = true;
  int rc = bart_run_batch(re_input, 1, transint, transit_out, transit_out_size, &status);
  if (rc == 0 && status == 0 && G.opt.savefiles) write_savefiles(re_input, transint);
  G.keep = saved_keep;
  G.knob_models = saved;
  if (rc != 0) return;
  // the reference exit()s where the batched path reports a per-model status
  if (status & REJ_SUMQ) fail("Sum of abundances of isotopes adds up to more than 1");
  if (status & REJ_TCIA) fail("A layer in the atmospheric model has a temperature outside the allowed "
                              "cross-section temperature range.");
  if (status & REJ_TGRID) {
    if (G.lbl) fail("A layer in the atmospheric model has a temperature outside the allowed TLI "
                    "temperature range [%.1f, %.1f] K.", G.tli.tmin, G.tli.tmax);
    fail("A layer in the atmospheric model has a temperature outside the "
         "opacity-grid temperature range [%g, %g] K.", G.og.temp.front(), G.og.temp.back());
  }
  if (status & REJ_FEWPTS) fail("Condition failed, less than 3 items for radial integration.");
  if (status & REJ_NOTOOMUCH) fail("Optical depth didn't reach limiting %g at some wavenumber.  Cannot "
                                   "use critical radius technique (-1).", G.opt.toomuch);
  API_END_VOID
}

void free_memory(void) {
  API_BEGIN
  reset_state();
  API_END_VOID
}

// =========================================================================================
// Part 2
void bart_set_error_mode(int mode) { g_error_mode = mode; }
const char *bart_last_error(void) { return g_error_msg; }
int bart_error_pending(void) { return g_error_pending ? 1 : 0; }
void bart_clear_error(void) { g_error_pending = false; g_error_msg[0] = 0; }

int bart_set_device(int ordinal) {
  API_BEGIN
  if (G.stream && ordinal != G.device) fail("bart_set_device must be called before transit_init");
  G.device = ordinal;
  return 0;
  API_END_INT
}
int bart_get_device(void) { return G.device; }

int bart_device_info(char *name, int name_len, int *sm_count, int *cc_major, int *cc_minor,
                     long long *l2_bytes, long long *hbm_bytes) {
  API_BEGIN
  ensure_device();
  cudaDeviceProp p;
  CUDA_OK(cudaGetDeviceProperties(&p, G.device));
  if (name && name_len > 0) snprintf(name, name_len, "%s", p.name);
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (cc_major) *cc_major = p.major;
  if (cc_minor) *cc_minor = p.minor;
  if (l2_bytes) *l2_bytes = p.l2CacheSize;
  if (hbm_bytes) *hbm_bytes = (long long)p.totalGlobalMem;
  return 0;
  API_END_INT
}

int bart_nlayers(void) { return G.dc.nlayer; }
int bart_nspecies(void) { return G.dc.nspec; }
int bart_ngridmol(void) { return G.dc.ngmol; }
int bart_ngridtemp(void) { return G.dc.ntemp; }
int bart_is_eclipse(void) { return G.dc.eclipse; }
long long bart_grid_bytes(void) {
  return (long long)G.og.nlayer * G.og.ntemp * G.og.nmol * G.og.nwave * 8;
}

int bart_set_batch_knobs(int nmodels, const double *refradius, const double *cloudtop,
                         const int *scat_flag, const double *scat_logext) {
  API_BEGIN
  ensure_device();
  Knobs &k = G.knobs;
  k.r0 = nullptr; k.cloudtop = nullptr; k.scat_flag = nullptr; k.scat_logext = nullptr;
  G.knob_models = 0;
  if (nmodels <= 0) return 0;
  if (refradius) { G.d_kr0.ensure(nmodels); CUDA_OK(cudaMemcpy(G.d_kr0.p, refradius, nmodels * 8, cudaMemcpyHostToDevice)); k.r0 = G.d_kr0.p; }
  if (cloudtop) { G.d_kcloud.ensure(nmodels); CUDA_OK(cudaMemcpy(G.d_kcloud.p, cloudtop, nmodels * 8, cudaMemcpyHostToDevice)); k.cloudtop = G.d_kcloud.p; }
  if (scat_flag) { G.d_kflag.ensure(nmodels); CUDA_OK(cudaMemcpy(G.d_kflag.p, scat_flag, nmodels * 4, cudaMemcpyHostToDevice)); k.scat_flag = G.d_kflag.p; }
  if (scat_logext) { G.d_klogext.ensure(nmodels); CUDA_OK(cudaMemcpy(G.d_klogext.p, scat_logext, nmodels * 8, cudaMemcpyHostToDevice)); k.scat_logext = G.d_klogext.p; }
  G.knob_models = nmodels;
  return 0;
  API_END_INT
}

int bart_run_batch_device(const double *d_profiles, int nmodels, int n_in, double *d_spectra,
                          int n_out, int *d_status) {
  API_BEGIN
  if (n_out < G.dc.nwave) fail("output holds %d values per model, %d needed", n_out, G.dc.nwave);
  if (n_out != G.dc.nwave) fail("bart_run_batch_device needs n_out == nwave (%d)", G.dc.nwave);
  run_models_device(d_profiles, nmodels, n_in, d_spectra);
  if (d_status)
    CUDA_OK(cudaMemcpyAsync(d_status, G.d_status.p, nmodels * sizeof(int), cudaMemcpyDeviceToDevice, G.stream));
  finish_stream();
  return 0;
  API_END_INT
}

int bart_run_batch(const double *profiles, int nmodels, int n_in, double *spectra, int n_out,
                   int *status) {
  API_BEGIN
  if (!G.init || G.opt.justOpacity) fail("Transit init not run, please initialize transit.");
  const int nw = G.dc.nwave;
  if (n_out < nw) fail("output holds %d values per model, %d needed", n_out, nw);
  if (nmodels <= 0) return 0;
  G.d_prof.ensure((size_t)nmodels * n_in);
  G.d_spec.ensure((size_t)nmodels * nw);
  prepare_batch(nmodels, n_in);
  // Small calls (run_transit = one model; a worker's handful of proposals): one stream, copies
  // through one pinned staging buffer (profiles in, spectra and status back), one synchronisation --
  // the three-stream pipeline below costs more in events and cross-stream hand-offs than such a
  // call has to overlap, and pageable buffers make every copy a staged, blocking one.
  const size_t lean_doubles = (size_t)nmodels * ((size_t)n_in + nw + 1);
  static const bool lean_on = [] { const char *e = getenv("BART_LEAN"); return !e || atoi(e) != 0; }();
  if (lean_on && lean_doubles * 8 <= (1u << 20)) {
    double *h_in = G.h_lean.ensure(lean_doubles), *h_out = h_in + (size_t)nmodels * n_in;
    int *h_st = reinterpret_cast<int *>(h_out + (size_t)nmodels * nw);
    memcpy(h_in, profiles, (size_t)nmodels * n_in * 8);
    CUDA_OK(cudaMemcpyAsync(G.d_prof.p, h_in, (size_t)nmodels * n_in * 8, cudaMemcpyHostToDevice, G.stream));
    launch_models(G.d_prof.p, 0, nmodels, nmodels, n_in, G.d_spec.p);
    CUDA_OK(cudaMemcpyAsync(h_out, G.d_spec.p, (size_t)nmodels * nw * 8, cudaMemcpyDeviceToHost, G.stream));
    if (status)
      CUDA_OK(cudaMemcpyAsync(h_st, G.d_status.p, nmodels * sizeof(int), cudaMemcpyDeviceToHost, G.stream));
    G.last_batch = nmodels;
    finish_stream();
    for (int m = 0; m < nmodels; m++) memcpy(spectra + (size_t)m * n_out, h_out + (size_t)m * nw, (size_t)nw * 8);
    if (status) memcpy(status, h_st, nmodels * sizeof(int));
    return 0;
  }
  // Software pipeline over chunks of the batch: H2D of chunk k+1 and D2H of chunk k-1 run on
  // their own streams (both copy engines) while chunk k computes.  Buffers are indexed by the
  // global model number, so chunks never alias.
  // Chunk schedule: small chunks at both ends keep the un-overlapped prologue (first H2D) and
  // epilogue (last D2H) short, 512-model chunks in the middle keep the kernels' tails rare.
  std::vector<int> sizes;
  if (G.keep || G.profile || G.lbl || nmodels < 1024) sizes.push_back(nmodels);
  else {
    const int ramp[2] = {128, 256};
    int left = nmodels;
    std::vector<int> head, tail;
    for (int k = 0; k < 2 && left >= 4 * ramp[k]; k++) { head.push_back(ramp[k]); tail.push_back(ramp[k]); left -= 2 * ramp[k]; }
    int nmid = std::max(1, left / 512);
    for (int k = 0; k < nmid; k++) sizes.push_back(left / nmid + (k < left % nmid ? 1 : 0));
    sizes.insert(sizes.begin(), head.begin(), head.end());
    sizes.insert(sizes.end(), tail.rbegin(), tail.rend());
  }
  const int nchunks = (int)sizes.size();
  while ((int)G.ev_pool.size() < 2 * nchunks + 1) {
    cudaEvent_t e;
    CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    G.ev_pool.push_back(e);
  }
  cudaEvent_t *ev_in = G.ev_pool.data(), *ev_k = G.ev_pool.data() + nchunks;
  cudaEvent_t ev_start = G.ev_pool[2 * nchunks];
  CUDA_OK(cudaEventRecord(ev_start, G.stream));             // order after earlier work on the stream
  CUDA_OK(cudaStreamWaitEvent(G.s_h2d, ev_start, 0));
  int off = 0;
  for (int c = 0; c < nchunks; c++) {
    const int cnt = sizes[c];
    CUDA_OK(cudaMemcpyAsync(G.d_prof.p + (size_t)off * n_in, profiles + (size_t)off * n_in,
                            (size_t)cnt * n_in * 8, cudaMemcpyHostToDevice, G.s_h2d));
    CUDA_OK(cudaEventRecord(ev_in[c], G.s_h2d));
    CUDA_OK(cudaStreamWaitEvent(G.stream, ev_in[c], 0));
    launch_models(G.d_prof.p + (size_t)off * n_in, off, cnt, nmodels, n_in, G.d_spec.p + (size_t)off * nw);
    CUDA_OK(cudaEventRecord(ev_k[c], G.stream));
    CUDA_OK(cudaStreamWaitEvent(G.s_d2h, ev_k[c], 0));
    if (n_out == nw)
      CUDA_OK(cudaMemcpyAsync(spectra + (size_t)off * nw, G.d_spec.p + (size_t)off * nw,
                              (size_t)cnt * nw * 8, cudaMemcpyDeviceToHost, G.s_d2h));
    else
      CUDA_OK(cudaMemcpy2DAsync(spectra + (size_t)off * n_out, (size_t)n_out * 8,
                                G.d_spec.p + (size_t)off * nw, (size_t)nw * 8, (size_t)nw * 8, cnt,
                                cudaMemcpyDeviceToHost, G.s_d2h));
    off += cnt;
  }
  if (status) {      // one small copy through pinned staging (a pageable target would block the loop)
    CUDA_OK(cudaMemcpyAsync(G.h_status.ensure(nmodels), G.d_status.p, nmodels * sizeof(int), cudaMemcpyDeviceToHost, G.s_d2h));
  }
  G.last_batch = nmodels;
  cudaError_t e = cudaStreamSynchronize(G.s_d2h);
  if (e != cudaSuccess) fail("CUDA execution failed: %s", cudaGetErrorString(e));
  finish_stream();
  if (status) memcpy(status, G.h_status.p, nmodels * sizeof(int));
  return 0;
  API_END_INT
}

int bart_set_filters(int nfilters, const int *start, const int *count, const double *weight,
                     const double *star, double rprs) {
  API_BEGIN
  ensure_device();
  if (nfilters <= 0) { G.nfilters = 0; return 0; }
  std::vector<int> off(nfilters);
  long long tot = 0;
  for (int f = 0; f < nfilters; f++) {
    if (start[f] < 0 || count[f] < 2 || start[f] + count[f] > (int)G.wn.size())
      fail("filter %d covers samples [%d, %d) outside the spectrum (%zu samples)", f, start[f],
           start[f] + count[f], G.wn.size());
    off[f] = (int)tot; tot += count[f];
  }
  G.d_fstart.ensure(nfilters); G.d_fcount.ensure(nfilters); G.d_foffset.ensure(nfilters);
  G.d_fweight.ensure(tot);
  CUDA_OK(cudaMemcpy(G.d_fstart.p, start, nfilters * 4, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(G.d_fcount.p, count, nfilters * 4, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(G.d_foffset.p, off.data(), nfilters * 4, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(G.d_fweight.p, weight, tot * 8, cudaMemcpyHostToDevice));
  G.have_star = star != nullptr;
  if (star) { G.d_fstar.ensure(tot); CUDA_OK(cudaMemcpy(G.d_fstar.p, star, tot * 8, cudaMemcpyHostToDevice)); }
  G.rprs2 = rprs * rprs;
  G.nfilters = nfilters;
  return 0;
  API_END_INT
}

int bart_nfilters(void) { return G.nfilters; }

int bart_set_energy_balance(int on, double e_in, double out_scale) {
  API_BEGIN
  if (on && !(e_in > 0 && out_scale > 0)) fail("bart_set_energy_balance: e_in and out_scale must be positive");
  G.eb_on = on != 0; G.eb_ein = e_in; G.eb_scale = out_scale;
  return 0;
  API_END_INT
}

int bart_energy_balance(const double *spectra, int nmodels, int nwave, int *rejected) {
  API_BEGIN
  if (!G.init || G.opt.justOpacity) fail("Transit init not run, please initialize transit.");
  if (!G.eb_on) fail("bart_set_energy_balance has not been called");
  if (nwave != G.dc.nwave) fail("bart_energy_balance: spectra have %d samples, expected %d", nwave, G.dc.nwave);
  if (nmodels <= 0) return 0;
  G.d_spec.ensure((size_t)nmodels * nwave);
  G.d_status.ensure(nmodels);
  CUDA_OK(cudaMemcpyAsync(G.d_spec.p, spectra, (size_t)nmodels * nwave * 8, cudaMemcpyHostToDevice, G.stream));
  CUDA_OK(cudaMemsetAsync(G.d_status.p, 0, nmodels * sizeof(int), G.stream));
  {
    KernelScope ks("energy_balance");
    launch_energy_balance(G.d_spec.p, G.d_wn.p, nwave, G.eb_scale, G.eb_ein, G.d_status.p, nmodels, G.stream);
    check_launch("energy_balance");
  }
  CUDA_OK(cudaMemcpyAsync(rejected, G.d_status.p, nmodels * sizeof(int), cudaMemcpyDeviceToHost, G.stream));
  finish_stream();
  return 0;
  API_END_INT
}

int bart_band_integrate(const double *spectra, int nmodels, int nwave, double *bandflux) {
  API_BEGIN
  if (nwave != (int)G.wn.size()) fail("bart_band_integrate: nwave %d != %zu", nwave, G.wn.size());
  G.d_spec.ensure((size_t)nmodels * nwave);
  G.d_band.ensure((size_t)nmodels * std::max(1, G.nfilters));
  CUDA_OK(cudaMemcpyAsync(G.d_spec.p, spectra, (size_t)nmodels * nwave * 8, cudaMemcpyHostToDevice, G.stream));
  band_device(G.d_spec.p, nmodels, nullptr, G.d_band.p);
  CUDA_OK(cudaMemcpyAsync(bandflux, G.d_band.p, (size_t)nmodels * G.nfilters * 8, cudaMemcpyDeviceToHost, G.stream));
  finish_stream();
  return 0;
  API_END_INT
}

int bart_bandflux_batch_device(const double *d_profiles, int nmodels, int n_in, double *d_bandflux,
                               int *d_status) {
  API_BEGIN
  G.d_spec.ensure((size_t)nmodels * G.dc.nwave);
  run_models_device(d_profiles, nmodels, n_in, G.d_spec.p);
  band_device(G.d_spec.p, nmodels, G.d_status.p, d_bandflux);
  if (d_status)
    CUDA_OK(cudaMemcpyAsync(d_status, G.d_status.p, nmodels * sizeof(int), cudaMemcpyDeviceToDevice, G.stream));
  finish_stream();
  return 0;
  API_END_INT
}

int bart_bandflux_batch(const double *profiles, int nmodels, int n_in, double *bandflux, int *status) {
  API_BEGIN
  if (!G.init || G.opt.justOpacity) fail("Transit init not run, please initialize transit.");
  if (nmodels <= 0) return 0;
  const int nw = G.dc.nwave;
  G.d_prof.ensure((size_t)nmodels * n_in);
  G.d_spec.ensure((size_t)nmodels * nw);
  G.d_band.ensure((size_t)nmodels * std::max(1, G.nfilters));
  prepare_batch(nmodels, n_in);
  // the profiles of chunk k+1 are copied in (copy stream) while chunk k computes; the band
  // integration and the small copy out follow the last chunk.  Chunks double from 256 models: the
  // only copy nothing hides is the first (2 MB), the copy engine then runs ahead of the kernels, and
  // the last chunk takes whatever is left -- at least half of the batch, so most of the batch runs
  // as one launch without the tail of a small grid
  std::vector<int> sizes;
  if (G.keep || G.profile || G.lbl || nmodels < 1024) sizes.push_back(nmodels);
  else {
    int left = nmodels;
    for (int c = 256; left - c >= 2 * c; c *= 2) { sizes.push_back(c); left -= c; }
    sizes.push_back(left);
  }
  const int nchunks = (int)sizes.size();
  while ((int)G.ev_pool.size() < nchunks + 1) {
    cudaEvent_t e;
    CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    G.ev_pool.push_back(e);
  }
  cudaEvent_t ev_start = G.ev_pool[nchunks];
  CUDA_OK(cudaEventRecord(ev_start, G.stream));
  CUDA_OK(cudaStreamWaitEvent(G.s_h2d, ev_start, 0));
  int off = 0;
  for (int c = 0; c < nchunks; c++) {
    const int cnt = sizes[c];
    CUDA_OK(cudaMemcpyAsync(G.d_prof.p + (size_t)off * n_in, profiles + (size_t)off * n_in,
                            (size_t)cnt * n_in * 8, cudaMemcpyHostToDevice, G.s_h2d));
    CUDA_OK(cudaEventRecord(G.ev_pool[c], G.s_h2d));
    CUDA_OK(cudaStreamWaitEvent(G.stream, G.ev_pool[c], 0));
    launch_models(G.d_prof.p + (size_t)off * n_in, off, cnt, nmodels, n_in, G.d_spec.p + (size_t)off * nw);
    off += cnt;
  }
  G.last_batch = nmodels;
  band_device(G.d_spec.p, nmodels, G.d_status.p, G.d_band.p);
  CUDA_OK(cudaMemcpyAsync(bandflux, G.d_band.p, (size_t)nmodels * G.nfilters * 8, cudaMemcpyDeviceToHost, G.stream));
  if (status)
    CUDA_OK(cudaMemcpyAsync(status, G.d_status.p, nmodels * sizeof(int), cudaMemcpyDeviceToHost, G.stream));
  finish_stream();
  return 0;
  API_END_INT
}

int bart_extinction_batch(const double *profiles, int nmodels, int n_in, double *ext_out, int what) {
  API_BEGIN
  if (!G.init || G.opt.justOpacity) fail("Transit init not run, please initialize transit.");
  DevConfig &c = G.dc;
  if (nmodels <= 0) return 0;
  const size_t n = (size_t)nmodels * c.nlayer * c.nwave;
  G.d_prof.ensure((size_t)nmodels * n_in);
  G.d_tabs.ensure((size_t)nmodels * c.lay.stride());
  G.d_status.ensure(nmodels);
  G.d_ext.ensure(n);
  CUDA_OK(cudaMemcpyAsync(G.d_prof.p, profiles, (size_t)nmodels * n_in * 8, cudaMemcpyHostToDevice, G.stream));
  Knobs k = effective_knobs(nmodels);
  if (G.lbl) prepare_batch(nmodels, n_in);
  { KernelScope ks("atm_prep");
    DevConfig cc = c;
    cc.lbl_model0 = 0;
    launch_atm_prep(cc, k, G.d_prof.p, n_in, G.d_tabs.p, G.d_status.p, nullptr, nmodels, G.stream); check_launch("atm_prep"); }
  if (G.lbl) lbl_extinction(G.d_prof.p, 0, nmodels, n_in);
  const int tiles = (c.nwave + kColThreads - 1) / kColThreads;
  int splits = 1;
  while ((long long)tiles * nmodels * splits < 148 * 8 && splits < c.nlayer) splits *= 2;
  { KernelScope ks("opacity_lookup");
    launch_extinction(c, G.d_tabs.p, G.d_ext.p, nmodels, what == 0 ? 1 : (what == 2 ? 2 : 0), splits, G.use_tma, G.stream);
    check_launch("opacity_lookup"); }
  if (ext_out)
    CUDA_OK(cudaMemcpyAsync(ext_out, G.d_ext.p, n * 8, cudaMemcpyDeviceToHost, G.stream));
  finish_stream();
  G.last_batch = nmodels;
  return 0;
  API_END_INT
}

// ---- memory helpers ----
void *bart_dev_alloc(long long bytes) {
  try { ensure_device(); } catch (BartError &) { return nullptr; }
  void *p = nullptr;
  if (cudaMalloc(&p, (size_t)bytes) != cudaSuccess) return nullptr;
  return p;
}
void bart_dev_free(void *p) { if (p) cudaFree(p); }
void *bart_host_alloc_pinned(long long bytes) {
  try { ensure_device(); } catch (BartError &) { return nullptr; }
  void *p = nullptr;
  if (cudaMallocHost(&p, (size_t)bytes) != cudaSuccess) return nullptr;
  return p;
}
void bart_host_free_pinned(void *p) { if (p) cudaFreeHost(p); }
int bart_memcpy_h2d(void *dst, const void *src, long long bytes) {
  API_BEGIN ensure_device();
  CUDA_OK(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyHostToDevice, G.stream));
  CUDA_OK(cudaStreamSynchronize(G.stream));
  return 0; API_END_INT
}
int bart_memcpy_d2h(void *dst, const void *src, long long bytes) {
  API_BEGIN ensure_device();
  CUDA_OK(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost, G.stream));
  CUDA_OK(cudaStreamSynchronize(G.stream));
  return 0; API_END_INT
}
int bart_sync(void) { API_BEGIN ensure_device(); finish_stream(); return 0; API_END_INT }

// ---- timing ----
int bart_timer_begin(void) {
  API_BEGIN ensure_device();
  CUDA_OK(cudaEventRecord(G.t0, G.stream));
  return 0; API_END_INT
}
double bart_timer_end(void) {
  try {
    ensure_device();
    CUDA_OK(cudaEventRecord(G.t1, G.stream));
    CUDA_OK(cudaEventSynchronize(G.t1));
    float ms = 0;
    CUDA_OK(cudaEventElapsedTime(&ms, G.t0, G.t1));
    return (double)ms;
  } catch (BartError &) { return -1.0; }
}
void bart_profile_enable(int on) { G.profile = on != 0; }
void bart_profile_reset(void) { G.stats.clear(); G.launches = 0; }
int bart_kernel_stats(int index, char *name, int name_len, long long *launches, double *ms) {
  if (index < 0 || index >= (int)G.stats.size()) return -1;
  auto it = G.stats.begin();
  std::advance(it, index);
  if (name && name_len > 0) snprintf(name, name_len, "%s", it->first.c_str());
  if (launches) *launches = it->second.launches;
  if (ms) *ms = it->second.ms;
  return 0;
}
long long bart_launch_count(void) { return G.launches; }
int bart_flush_l2(void) {
  API_BEGIN ensure_device();
  const size_t n = (size_t)(256u << 20) / 8;            // 256 MB > 126 MB L2
  G.d_flush.ensure(n);
  launch_fill(G.d_flush.p, n, 0.0, G.stream);
  check_launch("l2_flush");
  return 0; API_END_INT
}

// ---- introspection ----
void bart_debug_keep(int on) { G.keep = on != 0; }

long long bart_debug_get(const char *name, int model, double *out, long long capacity) {
  API_BEGIN
  if (!G.init) fail("not initialised");
  DevConfig &c = G.dc;
  const int nl = c.nlayer, nw = c.nwave;
  const std::string n = name;
  if (model < 0 || model >= G.last_batch) fail("bart_debug_get: model %d outside the last batch (%d)", model, G.last_batch);
  finish_stream();
  auto field = [&](int f, bool to_layer_order) -> long long {
    if (capacity < nl) fail("bart_debug_get: capacity too small");
    const int nf = c.lay.nf();
    std::vector<double> tmp((size_t)nl * nf);
    CUDA_OK(cudaMemcpy(tmp.data(), G.d_tabs.p + (size_t)model * c.lay.stride(), tmp.size() * 8,
                       cudaMemcpyDeviceToHost));
    for (int d = 0; d < nl; d++) out[to_layer_order ? nl - 1 - d : d] = tmp[(size_t)d * nf + f];
    return nl;
  };
  if (n == "radius") return field(TabLayout::RAD, true);
  if (n == "temp") return field(TabLayout::T, true);
  if (n == "scat") return field(TabLayout::SCAT, true);
  if (n == "cloud") return field(TabLayout::CLOUD, true);
  if (n == "simpson_a") return field(TabLayout::SA, false);
  if (n == "simpson_b") return field(TabLayout::SB, false);
  if (n == "simpson_c") return field(TabLayout::SC, false);
  if (n == "trapezoid") return field(TabLayout::TR, false);
  if (n == "table") {
    const long long cnt = c.lay.stride();
    if (capacity < cnt) fail("bart_debug_get: capacity too small");
    CUDA_OK(cudaMemcpy(out, G.d_tabs.p + (size_t)model * c.lay.stride(), cnt * 8, cudaMemcpyDeviceToHost));
    return cnt;
  }
  if (n == "tau") {          // [nwave][nlayer(depth)], like the reference's tau->t
    if (!G.keep || !G.d_tau.p) fail("bart_debug_get(tau): call bart_debug_keep(1) before the batch");
    const long long cnt = (long long)nw * nl;
    if (capacity < cnt) fail("bart_debug_get: capacity too small");
    CUDA_OK(cudaMemcpy(out, G.d_tau.p + (size_t)model * cnt, cnt * 8, cudaMemcpyDeviceToHost));
    return cnt;
  }
  if (n == "last") {
    if (!G.keep || !G.d_last.p) fail("bart_debug_get(last): call bart_debug_keep(1) before the batch");
    if (capacity < nw) fail("bart_debug_get: capacity too small");
    std::vector<int> tmp(nw);
    CUDA_OK(cudaMemcpy(tmp.data(), G.d_last.p + (size_t)model * nw, nw * 4, cudaMemcpyDeviceToHost));
    for (int i = 0; i < nw; i++) out[i] = tmp[i];
    return nw;
  }
  if (n == "ext") {          // after bart_extinction_batch: [nlayer][nwave]
    const long long cnt = (long long)nw * nl;
    if (!G.d_ext.p || capacity < cnt) fail("bart_debug_get(ext): no extinction batch or capacity too small");
    CUDA_OK(cudaMemcpy(out, G.d_ext.p + (size_t)model * cnt, cnt * 8, cudaMemcpyDeviceToHost));
    return cnt;
  }
  if (n == "status") {
    if (capacity < 1) fail("bart_debug_get: capacity too small");
    int s = 0;
    CUDA_OK(cudaMemcpy(&s, G.d_status.p + model, 4, cudaMemcpyDeviceToHost));
    out[0] = s;
    return 1;
  }
  fail("bart_debug_get: unknown name '%s'", name);
  return -1;
  API_END_INT
}

// ---- multi-GPU exchange: NCCL through dlopen (no link-time dependency) ----
typedef struct { char internal[128]; } nccl_uid_t;
typedef int (*fn_getuid)(nccl_uid_t *);
typedef int (*fn_initrank)(void **, int, nccl_uid_t, int);
typedef int (*fn_allgather)(const void *, void *, size_t, int, void *, cudaStream_t);
typedef int (*fn_destroy)(void *);
typedef const char *(*fn_errstr)(int);

static void *nccl_sym(const char *name) {
  if (!G.nccl_lib) {
    const char *cands[] = {"libnccl.so.2", "libnccl.so", nullptr};
    for (int i = 0; cands[i] && !G.nccl_lib; i++) G.nccl_lib = dlopen(cands[i], RTLD_NOW | RTLD_GLOBAL);
    if (!G.nccl_lib) fail("cannot load libnccl.so.2: %s", dlerror());
  }
  void *s = dlsym(G.nccl_lib, name);
  if (!s) fail("libnccl: symbol %s not found", name);
  return s;
}

// Peer windows: every rank allocates [2 slots][world][cap] doubles + arrival flags, the handles are
// exchanged with one ncclAllGather, and each rank maps the others' windows through CUDA IPC
// (NVLink/NVSwitch peer memory).  Any failure, on any rank, leaves every rank on the NCCL path.
static void setup_peer_window() {
  G.p2p = false;
  const char *env = getenv("BART_P2P");
  if (env && atoi(env) == 0) return;
  if (G.world < 2 || G.world > kMaxPeers) return;
  const long long cap = 1 << 18;                              // doubles per rank per slot (2 MiB)
  const size_t win_bytes = (size_t)2 * G.world * cap * 8;
  const size_t tail = 4096 + ((size_t)cap / kPeerGroup + 1) * 4;   // flags[world] | gen | done | err | group counters
  int ok = 1;
  if (!G.pw_base) {
    if (cudaMalloc((void **)&G.pw_base, win_bytes + tail) != cudaSuccess) { cudaGetLastError(); ok = 0; G.pw_base = nullptr; }
    else CUDA_OK(cudaMemset(G.pw_base, 0, win_bytes + tail));
  }
  struct Msg { cudaIpcMemHandle_t h; int ok; int pad[15]; };   // 128 bytes
  Msg mine; memset(&mine, 0, sizeof(mine));
  if (ok && cudaIpcGetMemHandle(&mine.h, G.pw_base) != cudaSuccess) { cudaGetLastError(); ok = 0; }
  mine.ok = ok;
  DevBuf<Msg> d_msg(1), d_all(G.world);
  std::vector<Msg> all(G.world);
  auto exchange = [&]() {
    CUDA_OK(cudaMemcpy(d_msg.p, &mine, sizeof(Msg), cudaMemcpyHostToDevice));
    int rc = ((fn_allgather)nccl_sym("ncclAllGather"))(d_msg.p, d_all.p, sizeof(Msg), 0 /*ncclInt8*/, G.nccl_comm, G.stream);
    if (rc != 0) fail("ncclAllGather failed: %s", ((fn_errstr)nccl_sym("ncclGetErrorString"))(rc));
    CUDA_OK(cudaStreamSynchronize(G.stream));
    CUDA_OK(cudaMemcpy(all.data(), d_all.p, sizeof(Msg) * G.world, cudaMemcpyDeviceToHost));
  };
  exchange();
  for (int r = 0; r < G.world; r++) ok = ok && all[r].ok;
  if (ok)
    for (int r = 0; r < G.world; r++) {
      if (r == G.rank) { G.pw_peer[r] = G.pw_base; continue; }
      if (cudaIpcOpenMemHandle(&G.pw_peer[r], all[r].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError(); G.pw_peer[r] = nullptr; ok = 0;
      }
    }
  mine.ok = ok;
  exchange();                                                 // everyone mapped everyone?
  for (int r = 0; r < G.world; r++) ok = ok && all[r].ok;
  if (!ok) { warn(1, "peer windows unavailable (CUDA IPC); using ncclAllGather\n"); return; }
  G.pw_cap = cap;
  G.pw_flags = (unsigned long long *)(G.pw_base + win_bytes);
  G.pw_gen = G.pw_flags + kMaxPeers;
  unsigned int *done = (unsigned int *)(G.pw_gen + 1);
  G.pw_err = (int *)(done + 2);
  PeerOut &po = G.pw;
  memset(&po, 0, sizeof(po));
  for (int r = 0; r < G.world; r++) {
    po.win[r] = (double *)G.pw_peer[r];
    po.flags[r] = (unsigned long long *)((char *)G.pw_peer[r] + win_bytes);
  }
  po.world = G.world; po.rank = G.rank; po.cap = cap; po.gen = G.pw_gen; po.done = done;
  po.grpcnt = (unsigned int *)(G.pw_base + win_bytes + 4096);
  G.p2p = true;
}

static void release_peer_window() {
  for (int r = 0; r < kMaxPeers; r++) {
    if (G.pw_peer[r] && G.pw_peer[r] != (void *)G.pw_base) cudaIpcCloseMemHandle(G.pw_peer[r]);
    G.pw_peer[r] = nullptr;
  }
  if (G.pw_base) { cudaFree(G.pw_base); G.pw_base = nullptr; }
  G.p2p = false;
}

int bart_comm_unique_id(char *id128) {
  API_BEGIN
  nccl_uid_t id;
  int rc = ((fn_getuid)nccl_sym("ncclGetUniqueId"))(&id);
  if (rc != 0) fail("ncclGetUniqueId failed: %s", ((fn_errstr)nccl_sym("ncclGetErrorString"))(rc));
  memcpy(id128, id.internal, 128);
  return 0;
  API_END_INT
}

int bart_comm_init(int rank, int world, const char *id128) {
  API_BEGIN
  ensure_device();
  nccl_uid_t id;
  memcpy(id.internal, id128, 128);
  int rc = ((fn_initrank)nccl_sym("ncclCommInitRank"))(&G.nccl_comm, world, id, rank);
  if (rc != 0) fail("ncclCommInitRank failed: %s", ((fn_errstr)nccl_sym("ncclGetErrorString"))(rc));
  G.rank = rank; G.world = world;
  setup_peer_window();
  return 0;
  API_END_INT
}

int bart_comm_p2p(void) { return G.p2p ? 1 : 0; }

// forward models -> band fluxes -> all ranks' band fluxes in d_all[world][nmodels*nfilters], every
// rank with the same nmodels.  Fused path: the band-integration kernel stores into the peers'
// windows; fallback: ncclAllGather.
int bart_bandflux_allgather_device(const double *d_profiles, int nmodels, int n_in,
                                   double *d_bandflux, double *d_all) {
  API_BEGIN
  if (G.world <= 1 || !G.nccl_comm) fail("bart_comm_init has not been called");
  const long long per_rank = (long long)nmodels * G.nfilters;
  const bool fused = p2p_usable(per_rank);
  G.d_spec.ensure((size_t)std::max(1, nmodels) * G.dc.nwave);
  run_models_device(d_profiles, nmodels, n_in, G.d_spec.p);
  band_device(G.d_spec.p, nmodels, G.d_status.p, d_bandflux, fused);
  if (fused) peer_gather(per_rank, d_all);
  else {
    int rc = ((fn_allgather)nccl_sym("ncclAllGather"))(d_bandflux, d_all, (size_t)per_rank, 8 /*ncclFloat64*/,
                                                        G.nccl_comm, G.stream);
    if (rc != 0) fail("ncclAllGather failed: %s", ((fn_errstr)nccl_sym("ncclGetErrorString"))(rc));
    G.launches++;
  }
  finish_stream();
  if (fused) check_peer_window("bart_bandflux_allgather_device");
  return 0;
  API_END_INT
}

int bart_comm_allgather(const double *d_send, double *d_recv, long long count_per_rank) {
  API_BEGIN
  if (!G.nccl_comm) fail("bart_comm_init has not been called");
  const int ncclFloat64 = 8;
  int rc = ((fn_allgather)nccl_sym("ncclAllGather"))(d_send, d_recv, (size_t)count_per_rank, ncclFloat64,
                                                      G.nccl_comm, G.stream);
  if (rc != 0) fail("ncclAllGather failed: %s", ((fn_errstr)nccl_sym("ncclGetErrorString"))(rc));
  G.launches++;
  finish_stream();
  return 0;
  API_END_INT
}

int bart_comm_finalize(void) {
  API_BEGIN
  if (G.nccl_comm) {
    // nobody may unmap a window a peer is still writing: agree first
    if (G.p2p) { finish_stream(); }
    ((fn_destroy)nccl_sym("ncclCommDestroy"))(G.nccl_comm); G.nccl_comm = nullptr;
  }
  release_peer_window();
  return 0;
  API_END_INT
}


// =========================================================================================
// Retrieval loop on the device (SURVEY.md 8f rows 1-2)

// replaces the input-converter set-up of code/BARTfunc.py:139-222
int bart_converter_init(int pt_type, int npt, const double *pt_args, int tint_thorngren,
                        const double *pressure_bar, const double *abundances, int nmolfit,
                        const int *imol, int nmetals, const int *imetals, int iH2, int iHe,
                        double tmin, double tmax, int nrad, int ncloud, int nray) {
  API_BEGIN
  if (!G.init || G.opt.justOpacity) fail("Transit init not run, please initialize transit.");
  const DevConfig &c = G.dc;
  ConvConfig cc{};
  const int want = pt_type == PT_ISO ? 1 : pt_type == PT_LINE ? 5 : pt_type == PT_ADIABATIC ? 3 :
                   pt_type == PT_MADHU_NOINV ? 5 : pt_type == PT_MADHU_INV ? 6 : pt_type == PT_PIETTE ? 8 : -1;
  if (want < 0)
    fail("unknown PT model %d (0 iso, 1 line, 2 adiabatic, 3 madhu_noinv, 4 madhu_inv, 5 piette)", pt_type);
  if (npt != want) fail("PT model %d takes %d parameters, got %d", pt_type, want, npt);
  if (nmolfit < 0 || nmolfit > kMaxGridMol) fail("too many fitted molecules (%d)", nmolfit);
  if (nmetals < 0 || nmetals > kMaxSpec) fail("too many metal species (%d)", nmetals);
  if (iH2 < 0 || iH2 >= c.nspec || iHe < 0 || iHe >= c.nspec) fail("H2/He species index out of range");
  if (nray < 0 || nray > 2 || nrad < 0 || nrad > 1 || ncloud < 0 || ncloud > 1) fail("bad knob counts");
  cc.pt_type = pt_type; cc.npt = npt; cc.nrad = nrad; cc.ncloud = ncloud; cc.nray = nray;
  cc.nmolfit = nmolfit; cc.nmetals = nmetals;
  cc.npars = npt + nrad + ncloud + (nray ? 1 : 0) + nmolfit;
  if (cc.npars > kMaxPars) fail("too many parameters (%d)", cc.npars);
  cc.nlayer = c.nlayer; cc.nspec = c.nspec;
  for (int i = 0; i < nmolfit; i++) {
    if (imol[i] < 0 || imol[i] >= c.nspec) fail("fitted molecule index %d out of range", imol[i]);
    cc.imol[i] = imol[i];
  }
  for (int i = 0; i < nmetals; i++) {
    if (imetals[i] < 0 || imetals[i] >= c.nspec) fail("metal index %d out of range", imetals[i]);
    cc.imetals[i] = imetals[i];
  }
  cc.iH2 = iH2; cc.iHe = iHe; cc.tmin = tmin; cc.tmax = tmax;
  if (pt_type == PT_LINE) {
    if (!pt_args) fail("PT_line needs pt_args = {R_star, T_star, T_int, sma, gravity}");
    cc.rstar = pt_args[0]; cc.tstar = pt_args[1]; cc.tint = pt_args[2]; cc.sma = pt_args[3];
    cc.grav = pt_args[4];
    if (tint_thorngren) {          // Thorngren et al. 2019, code/PT.py:671-676
      const double teq = sqrt(cc.rstar / (2.0 * cc.sma)) * cc.tstar;
      const double F = 4.0 * 5.6703744191844314e-08 * pow(teq, 4.0);
      cc.tint = 1.24 * teq * exp(-pow(log(F) - 0.14, 2.0) / 2.96);
    }
  }
  const int nl = c.nlayer, ns = c.nspec;
  std::vector<double> press(pressure_bar, pressure_bar + nl), base((size_t)ns * nl), ratio(nl);
  for (int l = 0; l < nl; l++) {
    for (int j = 0; j < ns; j++) base[(size_t)j * nl + l] = abundances[(size_t)l * ns + j];
    ratio[l] = abundances[(size_t)l * ns + iH2] / abundances[(size_t)l * ns + iHe];
  }
  upload(G.d_cpress, press); upload(G.d_cbase, base); upload(G.d_cratio, ratio);
  cc.press_bar = G.d_cpress.p; cc.base = G.d_cbase.p; cc.ratio = G.d_cratio.p;
  if (pt_type >= PT_MADHU_NOINV) {
    // the layer-smoothing models: Gaussian kernel of scipy.ndimage.gaussian_filter1d (truncate 4),
    // sigma = 4 layers (PT.py:372,581) or 0.3 dex (PT.py:810-811)
    cc.p_top = *std::min_element(press.begin(), press.end());
    cc.p_bot = *std::max_element(press.begin(), press.end());
    std::vector<double> x(nl);
    for (int l = 0; l < nl; l++) x[l] = log10(press[l]);
    double sigma = 4.0;
    if (pt_type == PT_PIETTE) {
      if (nl < 2) fail("PT_piette needs at least two layers");
      sigma = 0.3 / fabs(x[nl - 1] - x[nl - 2]);           // the reference's p runs top -> bottom
    }
    const int r = (int)(4.0 * sigma + 0.5);
    std::vector<double> w(2 * r + 1);
    const double c = -0.5 / (sigma * sigma);
    for (int k = -r; k <= r; k++) w[k + r] = exp(c * (double)(k * k));
    // numpy's pairwise sum (what phi_x.sum() evaluates; numpy/_core/src/umath/loops_utils.h.src)
    std::function<double(const double *, long)> pairwise = [&](const double *a, long n) -> double {
      if (n < 8) { double r = 0.0; for (long k = 0; k < n; k++) r += a[k]; return r; }
      if (n <= 128) {
        double acc[8];
        for (int j = 0; j < 8; j++) acc[j] = a[j];
        long k = 8;
        for (; k < n - (n % 8); k += 8) for (int j = 0; j < 8; j++) acc[j] += a[k + j];
        double r = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
        for (; k < n; k++) r += a[k];
        return r;
      }
      long n2 = n / 2;
      n2 -= n2 % 8;
      return pairwise(a, n2) + pairwise(a + n2, n - n2);
    };
    const double tot = pairwise(w.data(), (long)w.size());
    for (auto &v : w) v /= tot;
    upload(G.d_csmooth, w);
    cc.smooth_r = r; cc.smooth_w = G.d_csmooth.p;
    std::vector<int> seg(nl, 0);
    if (pt_type == PT_PIETTE) {
      // node layers on the reference's top -> bottom array (np.argmin: first occurrence)
      auto rev = [&](int i) { return press[nl - 1 - i]; };
      auto argmin_abs = [&](double target) {
        int best = 0;
        for (int i = 1; i < nl; i++) if (fabs(rev(i) - target) < fabs(rev(best) - target)) best = i;
        return best;
      };
      int top = 0, bot = 0;
      for (int i = 1; i < nl; i++) { if (rev(i) < rev(top)) top = i; if (rev(i) > rev(bot)) bot = i; }
      const int lay[8] = {top, argmin_abs(0.01), argmin_abs(0.1), argmin_abs(1.0), argmin_abs(3.2),
                          argmin_abs(10.0), argmin_abs(32.0), bot};
      for (int k = 0; k < 8; k++) cc.node_t[k] = x[nl - 1 - lay[k]];
      for (int k = 0; k < 7; k++)
        if (!(cc.node_t[k + 1] > cc.node_t[k]))
          fail("PT_piette: the pressure grid does not separate the eight node layers "
               "(top, 0.01, 0.1, 1, 3.2, 10, 32 bar, bottom)");
      for (int l = 0; l < nl; l++) {
        int k = 0;
        while (k < 6 && x[l] >= cc.node_t[k + 1]) k++;
        seg[l] = k;
      }
    }
    upload(G.d_cnodex, x);
    G.d_cnodeseg.ensure(nl);
    CUDA_OK(cudaMemcpy(G.d_cnodeseg.p, seg.data(), nl * sizeof(int), cudaMemcpyHostToDevice));
    cc.node_x = G.d_cnodex.p; cc.node_seg = G.d_cnodeseg.p;
  }
  cc.ready = 1;
  G.conv = cc;
  return 0;
  API_END_INT
}

int bart_converter_npars(void) { return G.conv.ready ? G.conv.npars : -1; }

int bart_profiles_from_params(const double *params, int nmodels, int npars, double *profiles,
                              int n_in, int *status, double *knobs_out) {
  API_BEGIN
  if (!G.conv.ready) fail("bart_converter_init has not been called");
  const ConvConfig &cc = G.conv;
  if (npars != cc.npars) fail("parameter vectors have %d entries, the converter expects %d", npars, cc.npars);
  const int need = (G.dc.nspec + 1) * G.dc.nlayer;
  if (n_in != need) fail("profiles hold %d values per model, %d needed", n_in, need);
  if (nmodels <= 0) return 0;
  G.d_cparams.ensure((size_t)nmodels * npars);
  G.d_prof.ensure((size_t)nmodels * n_in);
  G.d_cstatus.ensure(nmodels);
  G.d_kr0.ensure(nmodels); G.d_kcloud.ensure(nmodels); G.d_klogext.ensure(nmodels); G.d_kflag.ensure(nmodels);
  CUDA_OK(cudaMemcpyAsync(G.d_cparams.p, params, (size_t)nmodels * npars * 8, cudaMemcpyHostToDevice, G.stream));
  CUDA_OK(cudaMemsetAsync(G.d_prof.p, 0, (size_t)nmodels * n_in * 8, G.stream));
  ConvKnobs kn{G.d_kr0.p, G.d_kcloud.p, G.d_klogext.p, G.d_kflag.p};
  {
    KernelScope ks("convert_params");
    launch_convert_params(cc, G.d_cparams.p, npars, G.d_prof.p, n_in, G.d_cstatus.p, kn, nmodels, G.stream);
    check_launch("convert_params");
  }
  CUDA_OK(cudaMemcpyAsync(profiles, G.d_prof.p, (size_t)nmodels * n_in * 8, cudaMemcpyDeviceToHost, G.stream));
  if (status) CUDA_OK(cudaMemcpyAsync(status, G.d_cstatus.p, nmodels * sizeof(int), cudaMemcpyDeviceToHost, G.stream));
  finish_stream();
  if (knobs_out) {                       // [3][nmodels]: radius, cloudtop, scattering logext
    std::vector<double> tmp(nmodels);
    for (int k = 0; k < 3; k++) {
      const bool on = k == 0 ? cc.nrad : k == 1 ? cc.ncloud : cc.nray == 1;
      const double *src = k == 0 ? G.d_kr0.p : k == 1 ? G.d_kcloud.p : G.d_klogext.p;
      if (on) CUDA_OK(cudaMemcpy(knobs_out + (size_t)k * nmodels, src, nmodels * 8, cudaMemcpyDeviceToHost));
      else for (int m = 0; m < nmodels; m++) knobs_out[(size_t)k * nmodels + m] = 0.0;
    }
  }
  return 0;
  API_END_INT
}

int bart_bandflux_from_params_device(const double *d_params, int nmodels, int npars, double *d_bandflux,
                                     int *d_status) {
  API_BEGIN
  ensure_params_buffers(nmodels);
  params_to_bandflux_queued(d_params, nmodels, npars, d_bandflux);
  if (d_status && nmodels > 0)
    CUDA_OK(cudaMemcpyAsync(d_status, G.d_status.p, nmodels * sizeof(int), cudaMemcpyDeviceToDevice, G.stream));
  finish_stream();
  return 0;
  API_END_INT
}

int bart_bandflux_from_params(const double *params, int nmodels, int npars, double *bandflux, int *status) {
  API_BEGIN
  if (nmodels <= 0) return 0;
  ensure_params_buffers(nmodels);
  G.d_cparams.ensure((size_t)nmodels * npars);
  G.d_band.ensure((size_t)nmodels * G.nfilters);
  CUDA_OK(cudaMemcpyAsync(G.d_cparams.p, params, (size_t)nmodels * npars * 8, cudaMemcpyHostToDevice, G.stream));
  params_to_bandflux_queued(G.d_cparams.p, nmodels, npars, G.d_band.p);
  CUDA_OK(cudaMemcpyAsync(bandflux, G.d_band.p, (size_t)nmodels * G.nfilters * 8, cudaMemcpyDeviceToHost, G.stream));
  if (status) CUDA_OK(cudaMemcpyAsync(status, G.d_status.p, nmodels * sizeof(int), cudaMemcpyDeviceToHost, G.stream));
  finish_stream();
  return 0;
  API_END_INT
}

void bart_chain_block(int nchains, int world, int rank, int *lo, int *hi) {
  chain_block(nchains, world, rank, lo, hi);
}

// replaces the set-up and initial evaluation of MCcubed.mc.mcmc (mcmc.py:196-345) for walk='demc',
// for `nretr` independent retrievals in one loop: params[nretr][nchains][npars],
// data / uncert[nretr][ndata]; bounds, step sizes and priors shared
int bart_mcmc_init_ensemble(int nretr, int nchains, int npars, const double *params,
                            const double *pmin, const double *pmax, const double *stepsize,
                            const double *prior, const double *priorlow, int ndata,
                            const double *data, const double *uncert, double fgamma,
                            double fepsilon, int burnin) {
  API_BEGIN
  if (!G.conv.ready) fail("bart_converter_init has not been called");
  if (nretr < 1) fail("bart_mcmc_init: %d retrievals (need at least 1)", nretr);
  if (npars != G.conv.npars) fail("bart_mcmc_init: %d parameters, the converter expects %d", npars, G.conv.npars);
  if (ndata != G.nfilters) fail("bart_mcmc_init: %d data points but %d filters", ndata, G.nfilters);
  if (nchains < 3) fail("DE-MC needs at least 3 chains (got %d)", nchains);
  const int ntot = nretr * nchains;              // the flattened population
  McmcDev mc{};
  mc.nretr = nretr; mc.nchains = nchains; mc.npars = npars; mc.ndata = ndata; mc.burnin = burnin;
  mc.nold = 0;
  mc.fepsilon = fepsilon;
  for (int p = 0; p < npars; p++) {
    if (stepsize[p] > 0) mc.ifree[mc.nfree++] = p;
    else if (stepsize[p] < 0) {
      // a shared parameter copies parameter number -stepsize (1-based) (mcmc.py:307-308):
      // nextp[:, s] = nextp[:, -int(stepsize[s])-1]
      const int src = -(int)stepsize[p] - 1;
      if (src < 0 || src >= npars) fail("shared parameter %d points at %d", p, src);
      mc.share_dst[mc.nshare] = p; mc.share_src[mc.nshare] = src; mc.nshare++;
    }
    if (priorlow && priorlow[p] != 0) mc.iprior[mc.nprior++] = p;
  }
  if (mc.nfree < 1) fail("no free parameters");
  mc.gamma = fgamma * 2.4 / sqrt(2.0 * mc.nfree);
  auto up = [&](DevBuf<double> &b, const double *src, size_t n) -> double * {
    std::vector<double> v(n, 0.0);
    if (src) v.assign(src, src + n);
    upload(b, v);
    return b.p;
  };
  auto &mb = G.mcb;
  mc.pmin = up(mb.pmin, pmin, npars); mc.pmax = up(mb.pmax, pmax, npars);
  mc.prior = up(mb.prior, prior, npars); mc.priorlow = up(mb.priorlow, priorlow, npars);
  mc.data = up(mb.data, data, (size_t)nretr * ndata); mc.uncert = up(mb.uncert, uncert, (size_t)nretr * ndata);
  std::vector<double> p0(params, params + (size_t)ntot * npars);
  for (int g = 0; g < ntot; g++)
    for (int s = 0; s < mc.nshare; s++)
      p0[(size_t)g * npars + mc.share_dst[s]] = p0[(size_t)g * npars + mc.share_src[s]];
  mc.params = up(mb.params, p0.data(), p0.size());
  mc.nextp = up(mb.nextp, p0.data(), p0.size());
  mc.currchisq = up(mb.currchisq, nullptr, ntot); mc.nextchisq = up(mb.nextchisq, nullptr, ntot);
  mc.c2 = up(mb.c2, nullptr, ntot); mc.bestp = up(mb.bestp, nullptr, (size_t)nretr * npars);
  mc.bestchisq = up(mb.bestchisq, nullptr, nretr);
  mc.bestmodel = up(mb.bestmodel, nullptr, (size_t)nretr * ndata);
  mc.numaccept = up(mb.numaccept, nullptr, ntot);
  std::vector<int> zi((size_t)ntot * mc.nfree, 0);
  upload(mb.outbounds, zi); mc.outbounds = mb.outbounds.p;
  zi.assign(ntot, 0); upload(mb.outflag, zi); mc.outflag = mb.outflag.p;
  zi.assign(nretr, 0); upload(mb.iter, zi); mc.iter = mb.iter.p;
  G.mc = mc;
  G.mc_ztemplate = p0;
  G.mc_zsize = 0;
  chain_block(ntot, G.world, G.rank, &G.mc_lo, &G.mc_hi);
  G.mc_pad = ntot / G.world + (ntot % G.world ? 1 : 0);
  G.d_mcband.ensure((size_t)G.mc_pad * ndata);
  G.d_mcgather.ensure((size_t)G.mc_pad * ndata * G.world);
  CUDA_OK(cudaMemsetAsync(G.d_mcband.p, 0, (size_t)G.mc_pad * ndata * 8, G.stream));
  G.d_mccur.ensure((size_t)ntot * ndata);
  CUDA_OK(cudaMemsetAsync(G.d_mccur.p, 0, (size_t)ntot * ndata * 8, G.stream));
  G.mc.curmodel = G.d_mccur.p;
  G.d_mcallm.ensure((size_t)ntot * ndata);                 // the initial evaluation writes no trace
  G.mc.allmodel = G.d_mcallm.p;
  if (G.mc_graph) { cudaGraphExecDestroy(G.mc_graph); G.mc_graph = nullptr; }
  ensure_params_buffers(G.mc_hi - G.mc_lo);
  rank_barrier();
  mcmc_generation_queued(1);
  finish_stream();
  check_peer_window("bart_mcmc_init");
  G.mc_ready = true;
  return 0;
  API_END_INT
}

// replaces the set-up and initial evaluation of MCcubed.mc.mcmc (mcmc.py:196-345) for walk='demc':
// an ensemble of one
int bart_mcmc_init(int nchains, int npars, const double *params, const double *pmin,
                   const double *pmax, const double *stepsize, const double *prior,
                   const double *priorlow, int ndata, const double *data, const double *uncert,
                   double fgamma, double fepsilon, int burnin) {
  return bart_mcmc_init_ensemble(1, nchains, npars, params, pmin, pmax, stepsize, prior, priorlow,
                                 ndata, data, uncert, fgamma, fepsilon, burnin);
}

int bart_mcmc_nretr(void) { return G.mc_ready ? G.mc.nretr : 0; }

// MC3's resume=True for walk='demc' (mcmc.py:254-269): iterations of the previous run count towards
// burn-in and the savemodel trace continues from the previous run's last column
int bart_mcmc_resume(int nold, const double *curmodel) {
  API_BEGIN
  if (!G.mc_ready) fail("bart_mcmc_init has not been called");
  McmcDev &mc = G.mc;
  if (mc.nold != 0 || mc.chainsize != 0) fail("bart_mcmc_resume must come before the first bart_mcmc_run");
  if (nold < 0) fail("bart_mcmc_resume: nold = %d", nold);
  mc.nold = nold;
  if (curmodel)
    CUDA_OK(cudaMemcpyAsync(G.d_mccur.p, curmodel, (size_t)mc.nretr * mc.nchains * mc.ndata * 8,
                            cudaMemcpyHostToDevice, G.stream));
  finish_stream();
  return 0;
  API_END_INT
}

// replaces the generation loop of MCcubed.mc.mcmc (mcmc.py:518-625) for walk='demc'.  The random
// streams come from the caller in MC3's own shapes (mcmc.py:484-507), chainsize = niter.
int bart_mcmc_run(int niter, const double *support, const int *r1, const int *r2,
                  const double *unif, const double *ugamma) {
  API_BEGIN
  if (!G.mc_ready) fail("bart_mcmc_init has not been called");
  if (niter <= 0) return 0;
  McmcDev &mc = G.mc;
  const int nc = mc.nchains;
  const size_t n1 = (size_t)mc.nretr * nc * niter;       // every stream has nretr x niter x nchains entries
  for (int r = 0; r < mc.nretr; r++)
    for (int c = 0; c < nc; c++)
      for (int i = 0; i < niter; i++) {
        const size_t k = ((size_t)r * nc + c) * niter + i;
        if (r1[k] < 0 || r1[k] >= nc || r2[k] < 0 || r2[k] >= nc)
          fail("chain index out of range in r1/r2: retrieval %d, generation %d, chain %d (r1 %d, r2 %d, "
               "%d chains)", r, i, c, r1[k], r2[k], nc);
      }
  mc.nold += mc.chainsize;               // iterations of earlier calls count towards burn-in
  mc.chainsize = niter;
  mc.support = upload_queued(G.mcb.support, support, n1 * mc.nfree);
  mc.unif = upload_queued(G.mcb.unif, unif, n1);
  mc.ugamma = upload_queued(G.mcb.ugamma, ugamma, n1);
  mc.r1 = upload_queued(G.mcb.r1, r1, n1);
  mc.r2 = upload_queued(G.mcb.r2, r2, n1);
  mc.allparams = G.mcb.allparams.ensure(n1 * mc.nfree);
  G.d_mcallm.ensure(n1 * mc.ndata);
  mc.allmodel = G.d_mcallm.p;
  mc.walk = 0;
  mcmc_run_generations(niter);
  return 0;
  API_END_INT
}


// ---- snooker walk (BART's configured walk; ter Braak & Vrugt 2008 as in mcmc.py) ----
// (re)allocate the history for `rows` rows, keeping the filled ones; an unfilled row holds the
// chains' initial parameters (mcmc.py:419: Z[:, :, 0:mpars] = params; the generation loop only
// ever overwrites the free columns, 656)
static void snooker_reserve_rows(size_t rows) {
  McmcDev &mc = G.mc;
  if (rows <= G.mc_zcap) return;
  const size_t rowchains = (size_t)mc.nretr * mc.nchains;    // a row holds every retrieval's chains
  const size_t rowlen = rowchains * mc.npars;
  rows += rows / 2 + 16;
  DevBuf<double> nz, nc;
  nz.ensure(rows * rowlen); nc.ensure(rows * rowchains);
  std::vector<double> fill(rows * rowlen);
  for (size_t r = 0; r < rows; r++) std::copy(G.mc_ztemplate.begin(), G.mc_ztemplate.end(), fill.begin() + r * rowlen);
  CUDA_OK(cudaMemcpyAsync(nz.p, fill.data(), fill.size() * 8, cudaMemcpyHostToDevice, G.stream));
  CUDA_OK(cudaMemsetAsync(nc.p, 0, rows * rowchains * 8, G.stream));
  if (G.mc_zsize > 0) {
    CUDA_OK(cudaMemcpyAsync(nz.p, G.d_Z.p, (size_t)G.mc_zsize * rowlen * 8, cudaMemcpyDeviceToDevice, G.stream));
    CUDA_OK(cudaMemcpyAsync(nc.p, G.d_Zchisq.p, (size_t)G.mc_zsize * rowchains * 8, cudaMemcpyDeviceToDevice, G.stream));
  }
  CUDA_OK(cudaStreamSynchronize(G.stream));
  G.d_Z = std::move(nz); G.d_Zchisq = std::move(nc);
  G.mc_zcap = rows;
  mc.Z = G.d_Z.p; mc.Zchisq = G.d_Zchisq.p;
}

// replaces the Z set-up of MCcubed.mc.mcmc for walk='snooker' (mcmc.py:357-470): after
// bart_mcmc_init.  z0[hsize][nchains][nfree]: the M0 = hsize*nchains initial samples of the free
// parameters (the reference draws them uniformly in [pmin, pmax], 421-424; hsize must already be
// > nchains as mcmc.py:233-235 enforces); their models are evaluated here (429-447) and the best
// of them competes with the chains' best fit (449-470).
int bart_mcmc_snooker_init(int hsize, int thinning, const double *z0) {
  API_BEGIN
  if (!G.mc_ready) fail("bart_mcmc_init has not been called");
  McmcDev &mc = G.mc;
  if (hsize < 2) fail("snooker needs hsize >= 2 (got %d)", hsize);
  if (thinning < 1) fail("thinning must be >= 1 (got %d)", thinning);
  const int nc = mc.nchains, np = mc.npars, nr = mc.nretr, ntot = nr * nc;
  // fixed parameters of every Z sample are chain 0's of its retrieval (mcmc.py:425)
  for (int g = 0; g < ntot; g++)
    for (int p = 0; p < np; p++) {
      bool fixed = true;
      for (int f = 0; f < mc.nfree; f++) fixed &= mc.ifree[f] != p;
      for (int k = 0; k < mc.nshare; k++) fixed &= mc.share_dst[k] != p;
      if (fixed) G.mc_ztemplate[(size_t)g * np + p] = G.mc_ztemplate[(size_t)(g / nc) * nc * np + p];
    }
  G.mc_zsize = 0; G.mc_zcap = 0;
  snooker_reserve_rows((size_t)hsize + 64);
  // z0[nretr][hsize][nchains][nfree] -> rows [hsize][nretr][nchains][npars]
  std::vector<double> rows((size_t)hsize * ntot * np);
  for (int r = 0; r < nr; r++)
    for (int row = 0; row < hsize; row++)
      for (int c = 0; c < nc; c++) {
        const size_t g = (size_t)r * nc + c;
        double *dst = &rows[zidx(mc, row, r, c) * np];
        std::copy(&G.mc_ztemplate[g * np], &G.mc_ztemplate[g * np] + np, dst);
        const double *src = z0 + (((size_t)r * hsize + row) * nc + c) * mc.nfree;
        for (int f = 0; f < mc.nfree; f++) dst[mc.ifree[f]] = src[f];
      }
  CUDA_OK(cudaMemcpyAsync(mc.Z, rows.data(), rows.size() * 8, cudaMemcpyHostToDevice, G.stream));
  std::vector<int> zi(nr, hsize);
  upload(G.mcb.zsize, zi); mc.zsize = G.mcb.zsize.p;
  zi.assign(ntot, 0);
  upload(G.mcb.noproj, zi); mc.noproj = G.mcb.noproj.p;
  upload(G.mcb.slot, zi); mc.slot = G.mcb.slot.p;
  mc.zbest = G.mcb.zbest.ensure((size_t)nr * (1 + np + mc.ndata));
  mc.hsize = hsize; mc.thinning = thinning; mc.walk = 1;
  ensure_params_buffers(G.mc_hi - G.mc_lo);
  ModelMap mp{G.world, ntot / G.world, ntot % G.world, G.mc_pad};
  for (int row = 0; row < hsize; row++) {
    const double *models = mcmc_evaluate_queued(mc.Z + zidx(mc, row, 0, 0) * np);
    KernelScope ks("zrow_chisq");
    launch_zrow_chisq(mc, models, mp, row, row == hsize - 1, G.stream);
    check_launch("zrow_chisq");
  }
  finish_stream();
  check_peer_window("bart_mcmc_snooker_init");
  G.mc_zsize = hsize;
  return 0;
  API_END_INT
}

// replaces the generation loop of MCcubed.mc.mcmc for walk='snooker' (mcmc.py:518-660).  Random
// streams from the caller, in the order and shapes mcmc.py consumes them (chainsize = niter):
// support[niter][nchains][nfree], unif/ugamma[niter][nchains] (490-497); per generation i1, i2
// (flat indices into the first Zsize-1 rows x nchains, i1 != i2), iz (row < Zsize-1), ic (chain)
// [niter][nchains] (529-539); usnooker[usn_offset[niter]][nfree] the uniform(1.2, 2.2) factors
// of the chains with ugamma < 0.1, generation i owning rows usn_offset[i]..usn_offset[i+1]
// (545-556).  Zsize starts at hsize and grows by one after every generation with
// i % thinning == 0 (653-660).
int bart_mcmc_run_snooker(int niter, const double *support, const int *i1, const int *i2,
                          const int *iz, const int *ic, const double *usnooker,
                          const int *usn_offset, const double *unif, const double *ugamma) {
  API_BEGIN
  if (!G.mc_ready || G.mc_zsize < 2) fail("bart_mcmc_snooker_init has not been called");
  if (niter <= 0) return 0;
  McmcDev &mc = G.mc;
  const int nc = mc.nchains, nr = mc.nretr;
  // validate the indices against the history size each generation will see (every retrieval's
  // history grows on the same schedule); usn_offset[nretr][niter + 1] are absolute rows of usnooker,
  // the retrievals' factors one after the other
  int zs = G.mc_zsize;
  for (int r = 0; r < nr; r++) {
    zs = G.mc_zsize;
    const int *off = usn_offset + (size_t)r * (niter + 1);
    if (r > 0 && off[0] != off[-1])
      fail("usn_offset: retrieval %d starts at row %d, retrieval %d ended at row %d", r, off[0], r - 1, off[-1]);
    for (int i = 0; i < niter; i++) {
      int nsj = 0;
      for (int c = 0; c < nc; c++) {
        const size_t k = ((size_t)r * niter + i) * nc + c;
        const long long lim = (long long)(zs - 1) * nc;
        if (i1[k] < 0 || i1[k] >= lim || i2[k] < 0 || i2[k] >= lim || iz[k] < 0 || iz[k] >= zs - 1 ||
            ic[k] < 0 || ic[k] >= nc)
          fail("snooker index out of range: retrieval %d, generation %d, chain %d (history rows %d)", r,
               i, c, zs);
        nsj += ugamma[k] < 0.1;
      }
      if (off[i + 1] - off[i] != nsj || off[i] < 0)
        fail("usn_offset: retrieval %d, generation %d has %d snooker chains but %d rows of factors", r,
             i, nsj, off[i + 1] - off[i]);
      if ((mc.nold + mc.chainsize + i) % mc.thinning == 0) zs++;   // global iteration number
    }
  }
  snooker_reserve_rows((size_t)zs + 1);
  G.mc_zsize = zs;
  mc.nold += mc.chainsize;
  mc.chainsize = niter;
  // i1, i2, iz, ic packed in one buffer; usn_offset in another
  const size_t n1 = (size_t)nr * niter * nc;
  std::vector<int> packed(4 * n1);
  std::copy(i1, i1 + n1, packed.begin()); std::copy(i2, i2 + n1, packed.begin() + n1);
  std::copy(iz, iz + n1, packed.begin() + 2 * n1); std::copy(ic, ic + n1, packed.begin() + 3 * n1);
  const int *pk = upload_queued(G.d_snk_idx, packed.data(), packed.size());
  CUDA_OK(cudaStreamSynchronize(G.stream));
  mc.i1 = pk; mc.i2 = pk + n1; mc.iz = pk + 2 * n1; mc.ic = pk + 3 * n1;
  const size_t noff = (size_t)nr * (niter + 1);
  mc.usn_off = upload_queued(G.d_snk_off, usn_offset, noff);
  mc.usn = upload_queued(G.d_snk_usn, usnooker, (size_t)usn_offset[noff - 1] * mc.nfree);
  mc.support = upload_queued(G.mcb.support, support, n1 * mc.nfree);
  mc.unif = upload_queued(G.mcb.unif, unif, n1);
  mc.ugamma = upload_queued(G.mcb.ugamma, ugamma, n1);
  mc.allparams = G.mcb.allparams.ensure(n1 * mc.nfree);
  G.d_mcallm.ensure(n1 * mc.ndata);
  mc.allmodel = G.d_mcallm.p;
  mc.walk = 1;
  mcmc_run_generations(niter);
  return 0;
  API_END_INT
}

// results of the DE-MC loop: "allparams" [nchains][nfree][niter of the last run] (MC3's trace
// layout), "params" [nchains][npars], "currchisq", "numaccept" [nchains], "outbounds"
// [nchains][nfree], "bestp" [npars], "bestchisq" [1], "bestmodel" [ndata], "models" (band fluxes of
// the last generation, [nchains][ndata]), each behind a leading [nretr]; "Z" [nretr][Zsize]
// [nchains][npars], "Zchisq" [nretr][Zsize][nchains].  Returns the number of doubles written, or < 0.
long long bart_mcmc_get(const char *name, double *out, long long capacity) {
  API_BEGIN
  if (!G.mc_ready) fail("bart_mcmc_init has not been called");
  const McmcDev &mc = G.mc;
  const long long ntot = (long long)mc.nretr * mc.nchains;
  std::string n(name);
  const double *src = nullptr;
  long long cnt = 0;
  if (n == "allparams") { src = mc.allparams; cnt = ntot * mc.nfree * mc.chainsize; }
  else if (n == "allmodel") { src = mc.allmodel; cnt = ntot * mc.ndata * mc.chainsize; }
  else if (n == "params") { src = mc.params; cnt = ntot * mc.npars; }
  else if (n == "currchisq") { src = mc.currchisq; cnt = ntot; }
  else if (n == "numaccept") { src = mc.numaccept; cnt = ntot; }
  else if (n == "bestp") { src = mc.bestp; cnt = (long long)mc.nretr * mc.npars; }
  else if (n == "bestchisq") { src = mc.bestchisq; cnt = mc.nretr; }
  else if (n == "bestmodel") { src = mc.bestmodel; cnt = (long long)mc.nretr * mc.ndata; }
  else if (n == "Z" || n == "Zchisq") {
    // device rows [Zsize][nretr][nchains](...) -> retrieval-major [nretr][Zsize][nchains](...)
    if (!mc.Z) return 0;
    const long long w = n == "Z" ? mc.npars : 1, rowlen = ntot * w, blk = (long long)mc.nchains * w;
    cnt = (long long)G.mc_zsize * rowlen;
    if (cnt > capacity) fail("bart_mcmc_get(%s): capacity %lld < %lld", name, capacity, cnt);
    std::vector<double> tmp(cnt);
    if (cnt) CUDA_OK(cudaMemcpy(tmp.data(), n == "Z" ? mc.Z : mc.Zchisq, cnt * 8, cudaMemcpyDeviceToHost));
    for (int r = 0; r < mc.nretr; r++)
      for (int row = 0; row < G.mc_zsize; row++)
        std::copy(&tmp[row * rowlen + r * blk], &tmp[row * rowlen + r * blk] + blk,
                  out + ((long long)r * G.mc_zsize + row) * blk);
    return cnt;
  }
  else if (n == "outbounds") {
    cnt = ntot * mc.nfree;
    if (cnt > capacity) fail("bart_mcmc_get(%s): capacity %lld < %lld", name, capacity, cnt);
    std::vector<int> tmp(cnt);
    CUDA_OK(cudaMemcpy(tmp.data(), mc.outbounds, cnt * 4, cudaMemcpyDeviceToHost));
    for (long long i = 0; i < cnt; i++) out[i] = tmp[i];
    return cnt;
  } else if (n == "models") {
    cnt = ntot * mc.ndata;
    if (cnt > capacity) fail("bart_mcmc_get(%s): capacity %lld < %lld", name, capacity, cnt);
    const double *base = G.world > 1 ? G.d_mcgather.p : G.d_mcband.p;
    for (int r = 0; r < G.world; r++) {
      int lo, hi;
      chain_block((int)ntot, G.world, r, &lo, &hi);
      if (hi > lo)
        CUDA_OK(cudaMemcpy(out + (size_t)lo * mc.ndata, base + (size_t)r * G.mc_pad * mc.ndata,
                           (size_t)(hi - lo) * mc.ndata * 8, cudaMemcpyDeviceToHost));
    }
    return cnt;
  } else fail("bart_mcmc_get: unknown name '%s'", name);
  if (!src) return 0;
  if (cnt > capacity) fail("bart_mcmc_get(%s): capacity %lld < %lld", name, capacity, cnt);
  CUDA_OK(cudaMemcpy(out, src, cnt * 8, cudaMemcpyDeviceToHost));
  return cnt;
  API_END_INT
}

// ---- CLI support: one model from the atmosphere file's own profiles (transit.c:230-242 main) ----
int bart_cli_run(void) {
  API_BEGIN
  if (!G.init) fail("Transit init not run, please initialize transit.");
  if (G.opt.justOpacity) return 0;
  const int nl = G.atm.nlayer(), ns = G.atm.nspec(), nw = (int)G.wn.size();
  std::vector<double> in((size_t)(ns + 1) * nl), out(nw);
  for (int i = 0; i < nl; i++) in[i] = G.atm.temp[i];
  for (int j = 0; j < ns; j++)
    for (int i = 0; i < nl; i++) in[(size_t)(j + 1) * nl + i] = G.atm.q[(size_t)j * nl + i];
  // main() runs do_transit on the atmosphere as read: the file's own radius column, no hydrostatic
  // recomputation (that is reloadatm's, i.e. run_transit's, job)
  {
    DevBuf<double> d_rad;
    upload(d_rad, G.atm.radius);
    G.knobs.radius_file = d_rad.p;
    run_transit(in.data(), (int)in.size(), out.data(), nw);
    G.knobs.radius_file = nullptr;
  }
  if (bart_error_pending()) return -1;
  // printflux / printmod text format: eclipse.c:355-380, slantpath.c:510-555
  FILE *f = stdout;
  std::optional<File> file;
  const std::string &name = G.opt.outspec;
  if (!name.empty() && name != "-") {
    file.emplace(name.c_str(), "w");
    if (!*file) fail("Cannot open output file '%s'", name.c_str());
    f = *file;
  }
  const double wfct = 1.0;                       // wns.fct is always 1 (makesample.c:367)
  if (G.dc.eclipse) {
    fprintf(f, "#wvl [um]%*sFlux [erg/s/cm]\n", 6, " ");
    for (int w = 0; w < nw; w++) fprintf(f, "%-15.10g%-18.9g\n", 1e4 / (G.wn[w] / wfct), out[w]);
  } else {
    fprintf(f, "#wvl [um]        modulation\n");
    for (int w = 0; w < nw; w++) fprintf(f, "%-17.9g%-18.9g\n", 1e4 / (G.wn[w] / wfct), out[w]);
  }
  return 0;
  API_END_INT
}

// ---- builder entry points (builder.cu) ----
int bart_build_opacity_slice(int t_begin, int t_end, double *host_out) {
  API_BEGIN
  if (!G.init && !G.builder) fail("transit_init has not been called");
  ensure_device();
  builder_slice(G.builder, G.opt, G.atm, G.mol, G.tli, G.wn, G.stream, t_begin, t_end, host_out);
  return 0;
  API_END_INT
}

double bart_builder_phase_ms(const char *name) { return builder_phase_ms(G.builder.get(), name); }

long long bart_builder_stats(long long *nlines, long long *ngroups, long long *neval) {
  if (!G.builder) return -1;
  return builder_stats(G.builder.get(), nlines, ngroups, neval);
}

long long bart_line_bins(long long *iown_out, long long capacity) {
  API_BEGIN
  if (!G.builder) fail("the opacity-grid builder has not run in this process");
  return builder_line_bins(G.builder.get(), iown_out, capacity);
  API_END_INT
}

int bart_voigt_profile(int idop, int ilor, float *out, long long capacity, long long *halfsize) {
  API_BEGIN
  if (!G.builder) fail("the opacity-grid builder has not run in this process");
  return builder_profile(G.builder.get(), idop, ilor, out, capacity, halfsize);
  API_END_INT
}

}  // extern "C"
