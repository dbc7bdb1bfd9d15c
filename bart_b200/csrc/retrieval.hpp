// retrieval.hpp -- the retrieval loop around the forward model, on the device (retrieval.cu):
//   K-1 convert_params_kernel   input converter, code/BARTfunc.py:320-360 + code/PT.py:589-750
//   K7  demc_propose_kernel     DE-MC proposal, modules/MCcubed/MCcubed/mc/mcmc.py:524-575
//   K8  chisq_accept_kernel     chi-squared (src_c/chisq.c:111-142, include/stats.h:72-103),
//                               Metropolis rule, best fit, trace (mcmc.py:590-625), snooker
//                               Metropolis factor (603-609) and Z update (653-660)
//   K9  snooker_propose_kernel  DE-MC-with-snooker proposal from the sample history Z
//                               (ter Braak & Vrugt 2008; mcmc.py:527-561)
//   K10 zrow_chisq_kernel       chi-squared of the initial Z samples (mcmc.py:426-460)
//   K11 mcmc_draw_kernel,       the random streams of a seeded call from per-retrieval Philox
//       usn_scan_kernel,        keys (philox.cuh): MC3's constructions (mcmc.py:484-507,529-556),
//       usn_rows_kernel         other random numbers
//   K12 mcmc_retain_kernel      compaction of the loop state to a subset of its retrievals
#pragma once
#include "device.cuh"
#include <cuda_runtime.h>

namespace bart {

enum { REJ_TBOUNDS = 16, REJ_ABUND = 32, REJ_ENERGY = 128, REJ_PTMODEL = 256 };
enum { PT_ISO = 0, PT_LINE = 1, PT_ADIABATIC = 2, PT_MADHU_NOINV = 3, PT_MADHU_INV = 4, PT_PIETTE = 5 };
constexpr int kMaxPars = 64;

// Input converter set-up (BARTfunc.py:139-222).  Arrays live on the device.
struct ConvConfig {
  int ready;
  int pt_type, npt, nrad, ncloud, nray, nmolfit, nmetals, npars;
  int nlayer, nspec;
  int imol[kMaxGridMol];
  int imetals[kMaxSpec];
  int iH2, iHe;
  double tmin, tmax;
  double rstar, tstar, tint, sma, grav;    // PT_line arguments (BARTfunc.py:206-211); tint final
  const double *press_bar;                 // [nlayer] atmosphere-file order (bottom -> top)
  const double *base;                      // [nspec][nlayer] abundances of the atmosphere file
  const double *ratio;                     // [nlayer] H2/He
  // PT models that smooth over the layers (PT.py:157-586 Madhusudhan & Seager, 752-812 Piette):
  double p_top, p_bot;                     // min / max pressure (bar)
  int smooth_r;                            // Gaussian kernel radius, int(4 sigma + 0.5)
  const double *smooth_w;                  // [2 r + 1] normalised weights
  const double *node_x;                    // [nlayer] log10 p (Piette's interpolation abscissa)
  const int *node_seg;                     // [nlayer] knot interval of every layer
  double node_t[8];                        // Piette's eight knots (log10 p of the node layers)
};

// per-model knob arrays written by the converter (BARTfunc.py:350-360)
struct ConvKnobs {
  double *r0, *cloudtop, *scat_logext;
  int *scat_flag;
};

void launch_convert_params(const ConvConfig &cc, const double *params, int npars, double *profiles,
                           int n_in, int *status, const ConvKnobs &kn, int nmodels, cudaStream_t s);

// Energy-balance test of BARTfunc.py:366-383 on the spectra of a batch: a model whose outgoing
// energy trapz(spectrum, wn) * out_scale exceeds e_in gets REJ_ENERGY (its band fluxes then come
// out as -1, like every rejected model).  Models already rejected are left alone.
void launch_energy_balance(const double *spectra, const double *wn, int nwave, double out_scale,
                           double e_in, int *status, int nmodels, cudaStream_t s);

// DE-MC state (device pointers): an ensemble of `nretr` independent retrievals of `nchains` chains
// each, sharing the forward model, bounds, step sizes and priors.  The population is the flattened
// nretr x nchains models, g = r * nchains + c; arrays "per chain" below have that leading axis
// ([nretr][nchains]...), arrays "per retrieval" a leading [nretr].  nretr = 1 is one retrieval.
struct McmcDev {
  int nretr, nchains, npars, nfree, ndata, nprior, chainsize, burnin, nold;
  double gamma, fepsilon;
  int ifree[kMaxPars];
  int share_dst[kMaxPars], share_src[kMaxPars], nshare;
  int iprior[kMaxPars];
  const double *pmin, *pmax, *prior, *priorlow;   // shared, [npars]
  const double *data, *uncert;                    // per retrieval, [nretr][ndata]
  double *params, *nextp, *currchisq, *nextchisq, *c2;   // per chain
  double *bestp, *bestchisq, *bestmodel;          // per retrieval: [nretr][npars], [nretr], [nretr][ndata]
  double *numaccept, *allparams;                  // per chain; allparams[g][nfree][chainsize]
  // MC3's `savemodel` trace (mcmc.py:636-651): the model of every chain's CURRENT state after each
  // generation, allmodel[g][datum][iteration].  curmodel starts as zeros, like the reference's
  // `allmodel[~accepted,:,i+nold-1]` with i + nold - 1 = -1 at the first generation.
  double *curmodel, *allmodel;
  int *outbounds, *outflag;
  // generation counter of each retrieval [nretr], advanced by that retrieval's chi-squared CTA (the
  // only reader while it advances): generations replay as one captured graph
  int *iter;
  // random streams of this run, MC3's shapes (mcmc.py:484-507) behind a leading [nretr]
  const double *support;   // [nretr][chainsize][nchains][nfree]
  const int *r1, *r2;      // [nretr][nchains][chainsize], chain indices within the retrieval
  const double *unif;      // [nretr][chainsize][nchains]
  const double *ugamma;    // [nretr][chainsize][nchains]
  // walk = 1: snooker (mcmc.py:357-460,527-561,603-609,653-660)
  int walk, hsize, thinning;
  double *Z;               // [zcap][nretr][nchains][npars] sample history (zidx); rows carry the
                           // chains' initial non-free columns like the reference's (mcmc.py:419,425)
  double *Zchisq;          // [zcap][nretr][nchains]
  int *zsize;              // [nretr] rows filled so far (advance with the generations, all equal)
  double *zbest;           // [nretr][1 + npars + ndata] best initial Z sample: chisq, params, model
  const int *i1, *i2;      // [nretr][chainsize][nchains] flat (row, chain) indices into the retrieval's Z
  const int *iz, *ic;      // [nretr][chainsize][nchains]
  const double *usn;       // [sum of snooker chains][nfree] uniform(1.2, 2.2) factors, by retrieval
  const int *usn_off;      // [nretr][chainsize + 1] first row of generation i in usn
  int *noproj;             // per chain scratch: z == current state (mcmc.py:543)
  int *slot;               // per chain scratch: row of the chain's factors in usn
};

// row `row`, chain c of retrieval r in the history: one row holds every retrieval's chains, so a
// larger history is a prefix copy of a smaller one
BART_HD size_t zidx(const McmcDev &mc, int row, int r, int c) {
  return ((size_t)row * mc.nretr + r) * mc.nchains + c;
}

// where model g (of the flattened population) sits in the gathered band-flux buffer: rank blocks of
// `pad` rows
struct ModelMap { int world, base, extra, pad; };

// Random streams of a seeded call (bart_mcmc_run_seeded, philox.cuh), written into the buffers a
// host-stream call uploads into, in McmcDev's layouts.  DE-MC fills support / unif / ugamma / r1 / r2,
// snooker support / unif / ugamma / i1 / i2 / iz / ic / usn_off / usn (usn sized for every chain).
struct DrawArgs {
  const unsigned long long *keys;          // [nretr][2]
  const double *step;                      // [nfree] step sizes of the free parameters
  int nretr, nchains, nfree, niter, walk;
  long long it0;                           // global iteration of the call's generation 0
  int zs0, thinning;                       // snooker: history rows at generation 0, thinning
  double *support, *unif, *ugamma;
  int *r1, *r2, *i1, *i2, *iz, *ic, *usn_off;
  double *usn;
};
// draw kernel, then (snooker) the usn_off scan and the factor rows
void launch_mcmc_draws(const DrawArgs &d, cudaStream_t s);

// bart_mcmc_retain: every array of the loop state is laid out [outer][nretr][inner]; one entry
// gathers retrievals keep[0..nkeep) of one array into a new one laid out [outer][nkeep][inner].
// Outer rows >= `filled` are alike (unfilled history rows) and are all read from row `filled`.
struct RetainCopy {
  const void *src;
  void *dst;
  long long outer, filled, inner;          // inner: bytes of one retrieval's block
};
constexpr int kMaxRetainCopies = 32;
struct RetainArgs {
  RetainCopy c[kMaxRetainCopies];
  int n, nretr, nkeep;
  const int *keep;                         // device, [nkeep]
};
// one launch for every entry
void launch_mcmc_retain(const RetainArgs &a, cudaStream_t s);

// one warp per (retrieval, chain)
void launch_demc_propose(const McmcDev &mc, cudaStream_t s);
// the launches below run one CTA per retrieval
void launch_snooker_propose(const McmcDev &mc, cudaStream_t s);
// chi-squared of Z row `row` (models of its nretr x nchains samples); keeps each retrieval's running
// best in mc.zbest.
// last != 0: afterwards adopt zbest as the best fit when it beats the chains' (mcmc.py:462-470)
void launch_zrow_chisq(const McmcDev &mc, const double *models, ModelMap map, int row, int last,
                       cudaStream_t s);
// first = 1: initial state (mcmc.py:310-345): chi-squared of the current parameters, best fit
void launch_chisq_accept(const McmcDev &mc, const double *models, ModelMap map, int first,
                         cudaStream_t s);

}  // namespace bart
