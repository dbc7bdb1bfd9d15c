// retrieval.cu -- sm_100a kernels of the retrieval loop around the forward model (SURVEY.md 8f
// rows 1-2): a generation goes parameters -> profiles -> spectra -> band fluxes -> chi-squared ->
// Metropolis step without leaving the device.
//
//   convert_params_kernel  one CTA per proposal, thread <-> layer: temperature profile (PT_line of
//                          Line et al. 2013 with E_2 by series / continued fraction, PT_iso,
//                          PT_adiabatic; the layer-smoothing models PT_NoInversion / PT_Inversion of
//                          Madhusudhan & Seager 2009 and PT_piette, with scipy's Gaussian filter
//                          restated), abundance scaling 10^p, H2/He renormalisation, the two
//                          rejection tests, per-model radius / cloud-top / scattering knobs.
//                          Writes the profiles buffer in run_transit's layout, so atm_prep reads it
//                          unchanged.
//   demc_propose_kernel    warp <-> (retrieval, chain), lanes over parameters: DE-MC jump from two
//                          other chains' current states of the same retrieval, boundary clamp, shared
//                          parameters.  Products and sums are rounded separately (no FMA
//                          contraction) so chains are bit-identical to numpy.
//   chisq_accept_kernel    one CTA per retrieval: per-chain chi-squared with priors, Metropolis rule,
//                          state update, trace, running best fit (first-index argmin like numpy).
//   mcmc_draw_kernel       seeded runs only: the random streams of a call from per-retrieval Philox
//   (+ usn_scan, usn_rows) keys (philox.cuh), written where host streams are uploaded to.
//
// An ensemble of retrievals (McmcDev::nretr) is one flattened population g = r * nchains + c for the
// forward model; every per-retrieval step (partners, slot numbering, norm ratio, best fit, history)
// stays inside the retrieval's own chains and keeps the lone run's arithmetic and order, so
// retrieval r of an ensemble is bit-identical to the same retrieval run alone.
//
// These are latency-bound kernels over [nchains x npars] doubles: no roofline claim; they exist so
// that the per-generation host round trip (MPI scatter/gather in the reference) disappears.
#include "retrieval.hpp"
#include "dyn_smem.hpp"
#include "philox.cuh"
#include <cmath>

namespace bart {

// ---------------------------------------------------------------------------------------
// E_2(x): exponential integral of order 2 (scipy.special.expn(2, x) in code/PT.py:736).  A
// generation at MC3's 10-chain populations is bound by the longest dependent instruction chain of
// each of its kernels, and cephes' algorithm (power series for x <= 1, continued fraction above,
// each run to convergence) was most of the converter's: ~4700 instructions per warp.  Here
//   x <  1   E_2 = exp(-x) - x (h(x) - ln x), h(x) = E_1(x) + ln x = -gamma - sum_k (-x)^k / (k k!),
//            an entire function taken to degree kE2SeriesN - 1;
//   x >= 1   E_2 = F(x) exp(-x) / x, F(x) = x exp(x) E_2(x) (0.40 .. 1) from one polynomial per binade
//            2^k <= x < 2^(k+1), k = 0..9, in u = x / 2^(k-1) - 3 (Chebyshev interpolants in the monomial
//            basis)
// with tables computed at 60 digits by tools/gen_expint2_table.py: <= 1e-15 relative against mpmath
// on both branches (scipy's own expn is up to 3.5e-15 off just below x = 1: tests/test_expint2_table.py
// evaluates the tables on the CPU the way this function does), three orders inside what the profiles
// are held to against PT.py (1e-12, tests/test_gpu_retrieval.py).
#include "expint2_table.inc"
constexpr int kE2TableN = kE2SeriesN + kE2Intervals * kE2ChebN;
__device__ double g_e2_table[kE2TableN];        // series coefficients, then the binade polynomials
__device__ double expint2(double x, const double *tab) {
  const double MAXLOG = 7.09782712893383996843e2;
  if (!(x <= MAXLOG)) return x != x ? x : 0.0;
  if (x == 0.0) return 1.0;
  if (x >= 1.0) {
    const int hi = __double2hiint(x);
    const int k = (hi >> 20) - 1023;                                   // binade, 0..9
    const double scale = __hiloint2double((1024 - k) << 20, 0);        // 2^(1-k)
    const double u = fma(x, scale, -3.0);
    const double *t = tab + kE2SeriesN + k * kE2ChebN;
    double p = t[kE2ChebN - 1];
#pragma unroll
    for (int i = kE2ChebN - 2; i >= 0; i--) p = fma(p, u, t[i]);
    return p * exp(-x) / x;
  }
  double h = tab[kE2SeriesN - 1];
#pragma unroll
  for (int i = kE2SeriesN - 2; i >= 0; i--) h = fma(h, x, tab[i]);
  return exp(-x) - x * (h - log(x));
}

// eq. 14 of Line et al. 2013 (PT.py:719-737)
__device__ double line_xi(double gamma, double tau, const double *e2tab) {
  const double gt = gamma * tau;
  return (2.0 / 3) * (1 + (1. / gamma) * (1 + (0.5 * gamma * tau - 1) * exp(-gt)) +
                      gamma * (1 - 0.5 * (tau * tau)) * expint2(gt, e2tab));
}

// PT_line (PT.py:664-697) splits over a pair of adjacent lanes: each evaluates one of the two
// visible streams' xi (the expensive part), lane 0 of the pair combines them.  `half` = lane & 1.
// The quantities that depend on the parameters only are computed once per model (pt_line_consts):
// ptc = (kappa, gamma1, gamma2, Tint^4, Tirr^4).
enum { PTC_KAPPA = 0, PTC_G1 = 1, PTC_G2 = 2, PTC_TI4 = 3, PTC_TR4 = 4, PTC_N = 5 };
__device__ void pt_line_consts(const ConvConfig &cc, const double *par, int which, double *ptc) {
  if (which < 3) ptc[which] = pow(10.0, par[which]);
  else if (which == 3) ptc[PTC_TI4] = pow(cc.tint, 4.0);
  else if (which == 4) {
    const double tirr = par[4] * sqrt(cc.rstar / (2.0 * cc.sma)) * cc.tstar;
    ptc[PTC_TR4] = pow(tirr, 4.0);
  }
}
__device__ double pt_temperature(const ConvConfig &cc, const double *par, const double *ptc,
                                 const double *e2tab, double p_bar, int half) {
  if (cc.pt_type == PT_ISO) return par[0];
  if (cc.pt_type == PT_ADIABATIC) {             // PT.py:741-750
    const double p0 = pow(10.0, par[2]);
    return par[0] / (1 + (par[1] - 1) / par[1] * log(p0 / p_bar));
  }
  const double kappa = ptc[PTC_KAPPA], g = ptc[PTC_G1 + half];
  const double alpha = par[3];
  const double tau = kappa * (p_bar * 1e6) / cc.grav;
  const double xi_mine = line_xi(g, tau, e2tab);
  const double xi_other = __shfl_xor_sync(0xffffffffu, xi_mine, 1);
  const double xi1 = half ? xi_other : xi_mine, xi2 = half ? xi_mine : xi_other;
  const double ti4 = ptc[PTC_TI4], tr4 = ptc[PTC_TR4];
  // the fourth root as two square roots (each correctly rounded; PT.py's ** 0.25 is libm's pow)
  return sqrt(sqrt(0.75 * (ti4 * (2.0 / 3.0 + tau) + tr4 * (1 - alpha) * xi1 + tr4 * alpha * xi2)));
}

// Raw (unsmoothed) temperature of the smoothing PT models at one layer.  Arithmetic in the
// reference's order with separately rounded operations, so that only `log` (<= 1 ulp here,
// correctly rounded in glibc) can differ from PT.py.  *bad is set for the parameter sets the
// reference refuses (negative boundary temperatures, PT.py:337-340,543-545).
__device__ __forceinline__ double sq_rn(double x) { return __dmul_rn(x, x); }
__device__ double pt_raw_temperature(const ConvConfig &cc, const double *par, int l, int *bad) {
  const double p = cc.press_bar[l], p0 = cc.p_top;
  if (cc.pt_type == PT_MADHU_NOINV) {           // a1 a2 p1 p3 T3 (PT.py:384-586)
    const double a1 = par[0], a2 = par[1], p1 = par[2], p3 = par[3], T3 = par[4];
    const double T1 = __dsub_rn(T3, sq_rn(log(p3 / p1) / a2));
    const double T0 = __dsub_rn(T1, sq_rn(log(p1 / p0) / a1));
    if (T0 < 0 || T1 < 0 || T3 < 0) *bad = 1;
    if (p >= p0 && p < p1) return __dadd_rn(sq_rn(log(p / p0) / a1), T0);
    if (p >= p1 && p < p3) return __dadd_rn(sq_rn(log(p / p1) / a2), T1);
    if (p >= p3 && p <= cc.p_bot) return T3;
    return 0.0;
  }
  if (cc.pt_type == PT_MADHU_INV) {             // a1 a2 p1 p2 p3 T3 (PT.py:157-377)
    const double a1 = par[0], a2 = par[1], p1 = par[2], p2 = par[3], p3 = par[4], T3 = par[5];
    const double T2 = __dsub_rn(T3, sq_rn(log(p3 / p2) / a2));
    const double s10 = sq_rn(log(p1 / p0) / a1);
    const double T0 = __dsub_rn(__dadd_rn(T2, sq_rn(log(p1 / p2) / -a2)), s10);
    const double T1 = __dadd_rn(T0, s10);
    if (T0 < 0 || T1 < 0 || T2 < 0 || T3 < 0) *bad = 1;
    if (p >= p0 && p < p1) return __dadd_rn(sq_rn(log(p / p0) / a1), T0);
    if (p >= p1 && p < p2) return __dadd_rn(sq_rn(log(p / p2) / -a2), T2);
    if (p >= p2 && p < p3) return __dadd_rn(sq_rn(log(p / p2) / a2), T2);
    if (p >= p3 && p <= cc.p_bot) return T3;
    return 0.0;
  }
  // PT_piette (PT.py:752-812): T0 dTbot_32 dT32_10 dT10_0 dT0_1 dT1_01 dT01_001 dT001_top; knots
  // top, 10 mbar, 0.1, 1, 3.2, 10, 32 bar, bottom; degree-1 B-spline in log10 p (FITPACK fpbspl, k = 1)
  double Tn[8];
  Tn[4] = par[0];
  Tn[5] = __dadd_rn(par[0], par[3]);
  Tn[6] = __dadd_rn(Tn[5], par[2]);
  Tn[7] = __dadd_rn(Tn[6], par[1]);
  Tn[3] = __dsub_rn(par[0], par[4]);
  Tn[2] = __dsub_rn(Tn[3], par[5]);
  Tn[1] = __dsub_rn(Tn[2], par[6]);
  Tn[0] = __dsub_rn(Tn[1], par[7]);
  const int k = cc.node_seg[l];
  const double x = cc.node_x[l], t0 = cc.node_t[k], t1 = cc.node_t[k + 1];
  const double f = 1.0 / __dsub_rn(t1, t0);
  return __dadd_rn(__dmul_rn(Tn[k], __dmul_rn(f, __dsub_rn(t1, x))),
                   __dmul_rn(Tn[k + 1], __dmul_rn(f, __dsub_rn(x, t0))));
}

// scipy.ndimage.gaussian_filter1d(T, sigma, mode='nearest') at layer l: the symmetric branch of
// NI_Correlate1D -- centre term first, then the pairs from the outermost inwards, the ends
// extended with the end values.  Symmetric in the layer order, so it does not matter that the
// reference smooths the top -> bottom array (BARTfunc.py:176,321).
__device__ double smooth_nearest(const ConvConfig &cc, const double *T, int l) {
  const int r = cc.smooth_r, nl = cc.nlayer;
  double t = __dmul_rn(T[l], cc.smooth_w[r]);
  for (int j = -r; j < 0; j++) {
    const int a = max(l + j, 0), b = min(l - j, nl - 1);
    t = __dadd_rn(t, __dmul_rn(__dadd_rn(T[a], T[b]), cc.smooth_w[r + j]));
  }
  return t;
}

constexpr int kConvThreads = 256;               // two lanes per layer
// `staged`: the arrays of the set-up (pressures, base abundances, H2/He ratio) come in through one
// round of coalesced loads into shared memory and the profile is assembled there and written out as
// one stream -- at MC3's population sizes the kernel is a chain of memory latencies (the abundance
// loop alone was a dependent global load + store per species).  Same arithmetic, same order.
// Shared-memory doubles: [nlayer] raw temperatures | staged: press[nl], ratio[nl], base[nspec][nl],
// profile[(1 + nspec)][nl]
__global__ void __launch_bounds__(kConvThreads)
convert_params_kernel(ConvConfig cc, const double *__restrict__ params, int npars,
                      double *__restrict__ profiles, int n_in, int *__restrict__ status,
                      ConvKnobs kn, int nmodels, int staged) {
  const int m = blockIdx.x;
  if (m >= nmodels) return;
  extern __shared__ double s_T[];               // [nlayer] raw temperatures (smoothing PT models)
  __shared__ int s_bad;
  __shared__ double s_par[kMaxPars];
  __shared__ double s_fac[kMaxPars];            // 10^p of the abundance parameters
  __shared__ double s_ptc[PTC_N];               // per-model constants of PT_line
  __shared__ double s_e2[kE2TableN];
  if (threadIdx.x == 0) s_bad = 0;
  const bool line = cc.pt_type == PT_LINE;
  if (line)
    for (int i = threadIdx.x; i < kE2TableN; i += blockDim.x) s_e2[i] = g_e2_table[i];
  const int nl = cc.nlayer;
  // either scattering model takes one parameter slot (polar, nray 2, leaves its value unused): the
  // molecules' factors follow it (BARTfunc.py:333-338)
  const int off = cc.npt + cc.nrad + cc.ncloud + (cc.nray ? 1 : 0);
  double *gout = profiles + (size_t)m * n_in;
  const double *press = cc.press_bar, *ratio_a = cc.ratio, *base = cc.base;
  double *out = gout;
  if (staged) {
    double *s_press = s_T + nl, *s_ratio = s_press + nl, *s_base = s_ratio + nl;
    double *s_prof = s_base + (size_t)cc.nspec * nl;
    for (int i = threadIdx.x; i < nl; i += blockDim.x) { s_press[i] = cc.press_bar[i]; s_ratio[i] = cc.ratio[i]; }
    for (int i = threadIdx.x; i < cc.nspec * nl; i += blockDim.x) s_base[i] = cc.base[i];
    press = s_press; ratio_a = s_ratio; base = s_base; out = s_prof;
  }
  for (int i = threadIdx.x; i < npars; i += blockDim.x) {
    const double v = params[(size_t)m * npars + i];
    s_par[i] = v;
    if (i >= off && i - off < cc.nmolfit) s_fac[i - off] = pow(10.0, v);
  }
  // PT_line's per-model constants, one thread each (the last warp: the first ones hold the pows above)
  if (line && threadIdx.x >= kConvThreads - PTC_N)
    pt_line_consts(cc, params + (size_t)m * npars, threadIdx.x - (kConvThreads - PTC_N), s_ptc);
  __syncthreads();
  int bad = 0;
  const bool smoothed = cc.pt_type >= PT_MADHU_NOINV;
  if (smoothed) {
    int refused = 0;
    for (int l = threadIdx.x; l < nl; l += blockDim.x) s_T[l] = pt_raw_temperature(cc, s_par, l, &refused);
    // The reference catches the ValueError and carries on with the profile of the worker's PREVIOUS
    // proposal ("FINDME: what to do here?", BARTfunc.py:323-325); a batch has no previous proposal,
    // the model is rejected
    if (refused) bad |= REJ_PTMODEL;
    __syncthreads();
  }
  const int half = threadIdx.x & 1;
  // every lane of a warp runs the same number of passes (the pair exchange is a warp shuffle)
  const int npass = (nl + kConvThreads / 2 - 1) / (kConvThreads / 2);
  for (int pass = 0; pass < npass; pass++) {
    const int l = pass * (kConvThreads / 2) + (threadIdx.x >> 1);
    const bool live = l < nl;
    const double T = smoothed ? smooth_nearest(cc, s_T, live ? l : nl - 1)
                              : pt_temperature(cc, s_par, s_ptc, s_e2, press[live ? l : nl - 1], half);
    if (!live || half) continue;
    if (!(T >= cc.tmin) || !(T <= cc.tmax)) bad |= REJ_TBOUNDS;   // also catches NaN
    out[l] = T;
    // scaled abundances and the metal sum in the reference's order (BARTfunc.py:333-338)
    double metals = 0.0;
    for (int j = 0; j < cc.nspec; j++) {
      double a = base[(size_t)j * nl + l];
      for (int k = 0; k < cc.nmolfit; k++)
        if (cc.imol[k] == j) a = a * s_fac[k];
      if (j != cc.iH2 && j != cc.iHe) out[(size_t)(j + 1) * nl + l] = a;
    }
    for (int k = 0; k < cc.nmetals; k++) {
      const double a = out[(size_t)(cc.imetals[k] + 1) * nl + l];
      metals = k == 0 ? a : metals + a;
    }
    const double q = 1.0 - metals;
    if (q < 0.0) bad |= REJ_ABUND;
    const double ratio = ratio_a[l];
    out[(size_t)(cc.iH2 + 1) * nl + l] = ratio * q / (1.0 + ratio);
    out[(size_t)(cc.iHe + 1) * nl + l] = q / (1.0 + ratio);
  }
  if (bad) atomicOr(&s_bad, bad);
  __syncthreads();
  if (staged) {
    const int nprof = (cc.nspec + 1) * nl;
    for (int i = threadIdx.x; i < nprof; i += blockDim.x) gout[i] = out[i];
  }
  if (threadIdx.x == 0) {
    // the temperature test comes first and wins (BARTfunc.py:327-330 before 339-344)
    status[m] = (s_bad & REJ_PTMODEL) ? REJ_PTMODEL : (s_bad & REJ_TBOUNDS) ? REJ_TBOUNDS : s_bad;
    int c = cc.npt;
    if (cc.nrad) kn.r0[m] = s_par[c++];
    if (cc.ncloud) kn.cloudtop[m] = s_par[c++];
    if (cc.nray == 1) { kn.scat_flag[m] = 1; kn.scat_logext[m] = s_par[c]; }
    else if (cc.nray == 2) { kn.scat_flag[m] = 2; kn.scat_logext[m] = 0.0; }
  }
}

void launch_convert_params(const ConvConfig &cc, const double *params, int npars, double *profiles,
                           int n_in, int *status, const ConvKnobs &kn, int nmodels, cudaStream_t s) {
  if (nmodels <= 0) return;
  static bool table_ready = false;
  if (!table_ready) {
    double h[kE2TableN];
    for (int i = 0; i < kE2SeriesN; i++) h[i] = kE2SeriesHost[i];
    for (int i = 0; i < kE2Intervals * kE2ChebN; i++) h[kE2SeriesN + i] = kE2ChebHost[i];
    // on the launch stream and awaited: `h` is pageable, and the kernel below runs on `s`, which
    // does not synchronise with the legacy stream a plain cudaMemcpyToSymbol uses
    cudaMemcpyToSymbolAsync(g_e2_table, h, sizeof(h), 0, cudaMemcpyHostToDevice, s);
    cudaStreamSynchronize(s);
    table_ready = true;
  }
  size_t smem = ((size_t)cc.nlayer * 3 + (size_t)cc.nspec * cc.nlayer * 2 + cc.nlayer) * sizeof(double);
  const int staged = smem <= 96 * 1024;
  if (!staged) smem = (size_t)cc.nlayer * sizeof(double);
  if (!allow_dyn_smem<convert_params_kernel>(smem)) return;
  convert_params_kernel<<<nmodels, kConvThreads, smem, s>>>(cc, params, npars, profiles, n_in, status, kn, nmodels, staged);
}

// ---------------------------------------------------------------------------------------
// Energy balance (BARTfunc.py:366-383): e_out = np.trapz(spectrum, specwn) * 4 (100 Rp)^2 against
// e_in = sigma Ts^4 Rs^2 pi Rp^2 / a^2 * 1e7 (computed once on the host).  One CTA per model,
// fixed-shape reduction (deterministic); the comparison is a threshold test, so the summation order
// (numpy's pairwise sum in the reference) matters only for a model exactly on the threshold.
__global__ void __launch_bounds__(256)
energy_balance_kernel(const double *__restrict__ spectra, const double *__restrict__ wn, int nwave,
                      double out_scale, double e_in, int *__restrict__ status, int nmodels) {
  const int m = blockIdx.x;
  if (m >= nmodels || status[m] != 0) return;               // CTA-uniform
  const double *sp = spectra + (size_t)m * nwave;
  double acc = 0.0;
  for (int i = threadIdx.x; i < nwave - 1; i += blockDim.x)
    acc += (wn[i + 1] - wn[i]) * (sp[i + 1] + sp[i]) / 2.0;
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  __shared__ double s_part[8];
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; w++) t += s_part[w];
    if (t * out_scale > e_in) status[m] = REJ_ENERGY;
  }
}

void launch_energy_balance(const double *spectra, const double *wn, int nwave, double out_scale,
                           double e_in, int *status, int nmodels, cudaStream_t s) {
  if (nmodels <= 0) return;
  energy_balance_kernel<<<nmodels, 256, 0, s>>>(spectra, wn, nwave, out_scale, e_in, status, nmodels);
}

// ---------------------------------------------------------------------------------------
// DE-MC proposal (mcmc.py:524-575): jump = gamma1 (x_r1 - x_r2) + fepsilon * support
// One warp per (retrieval, chain), lanes over the free parameters: the loads of a jump (two other chains' states,
// the support draw, the bounds) go out side by side instead of as one dependent round trip per
// parameter (at MC3's population sizes the kernel's time is its chain of memory latencies).
__global__ void __launch_bounds__(256) demc_propose_kernel(McmcDev mc) {
  const int lane = threadIdx.x & 31;
  const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // (retrieval, chain) flattened
  const int nc = mc.nchains;
  if (g >= mc.nretr * nc) return;               // whole warps
  const int r = g / nc, c = g - r * nc;
  const int i = mc.iter[r];
  const int np = mc.npars;
  const double *cur = mc.params + (size_t)g * np;
  double *nx = mc.nextp + (size_t)g * np;
  const int ra = mc.r1[(size_t)g * mc.chainsize + i], rb = mc.r2[(size_t)g * mc.chainsize + i];
  const size_t k = ((size_t)r * mc.chainsize + i) * nc + c;    // this chain's entry of generation i
  const double ug = mc.ugamma[k];
  const double *a = mc.params + ((size_t)r * nc + ra) * np;
  const double *b = mc.params + ((size_t)r * nc + rb) * np;
  const double gm = ug < 0.1 ? 0.98 : mc.gamma;
  const double *sup = mc.support + k * mc.nfree;
  int out = 0;
  for (int f = lane; f < mc.nfree; f += 32) {
    const int p = mc.ifree[f];
    const double ap = a[p], bp = b[p], cp = cur[p], sf = sup[f], lo = mc.pmin[p], hi = mc.pmax[p];
    const int ob = mc.outbounds[(size_t)g * mc.nfree + f];
    const double jump = __dadd_rn(__dmul_rn(gm, __dsub_rn(ap, bp)), __dmul_rn(mc.fepsilon, sf));
    double v = __dadd_rn(cp, jump);
    const int o = (v < lo) || (v > hi);
    out |= o;
    mc.outbounds[(size_t)g * mc.nfree + f] = ob + o;
    if (v < lo) v = lo;
    if (v > hi) v = hi;
    nx[p] = v;
  }
  out = __any_sync(0xffffffffu, out) ? 1 : 0;
  __syncwarp();                                 // the lanes' nx[] are visible to lane 0
  if (lane == 0) {
    for (int s = 0; s < mc.nshare; s++) nx[mc.share_dst[s]] = nx[mc.share_src[s]];
    mc.outflag[g] = out;
  }
}

void launch_demc_propose(const McmcDev &mc, cudaStream_t s) {
  const int threads = 256;                      // 8 chains per CTA
  const int warps = mc.nretr * mc.nchains;
  demc_propose_kernel<<<(warps * 32 + threads - 1) / threads, threads, 0, s>>>(mc);
}

// ---------------------------------------------------------------------------------------
// numpy's pairwise summation (numpy/_core/src/umath/loops_utils.h.src, n <= 128), i.e. what
// np.sum(x, axis=1) computes along a contiguous axis: the snooker projection's dot products
// (mcmc.py:551-556) are reproduced bit for bit
__device__ double np_pairwise_sum(const double *a, int n) {
  if (n < 8) {
    double r = 0.0;
    for (int k = 0; k < n; k++) r = __dadd_rn(r, a[k]);
    return r;
  }
  double r[8];
  for (int j = 0; j < 8; j++) r[j] = a[j];
  int k = 8;
  for (; k < n - (n % 8); k += 8)
    for (int j = 0; j < 8; j++) r[j] = __dadd_rn(r[j], a[k + j]);
  double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                         __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
  for (; k < n; k++) res = __dadd_rn(res, a[k]);
  return res;
}

// Snooker proposal (mcmc.py:527-575).  Per chain: two history samples z1 = Z[i1], z2 = Z[i2] and
// a projection anchor z = Z[iz][ic].  With probability 0.9 (ugamma >= 0.1) a DE-MC jump
// gamma (z1 - z2) + fepsilon support; otherwise a snooker jump u (zp1 - zp2)/|x - z|^2 (x - z)
// along x - z (zp = projections of z1, z2), or u (z2 - z1) when z coincides with the chain's
// state.  The uniform factors u come in the reference from two calls whose sizes depend on the
// states (unprojected chains first): `slot` reproduces that assignment.
// One CTA per retrieval (the slot numbering below is one ordered pass over its chains); a warp per chain with
// lanes over the parameters, like demc_propose_kernel: the loads of a jump go out side by side and the
// projection's three dot products are numpy's pairwise sums (np_pairwise_sum, every lane the same
// sequence) over the warp's products in shared memory.
constexpr int kSnkThreads = 512;
__global__ void __launch_bounds__(kSnkThreads) snooker_propose_kernel(McmcDev mc) {
  __shared__ double s_dz[kSnkThreads / 32][kMaxPars], s_t[3][kSnkThreads / 32][kMaxPars];
  const int r = blockIdx.x;                     // retrieval
  const int i = mc.iter[r];
  const int np = mc.npars, nc = mc.nchains;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const size_t gen = ((size_t)r * mc.chainsize + i) * nc;   // generation i of retrieval r in the streams
  const int *gi1 = mc.i1 + gen, *gi2 = mc.i2 + gen;
  const int *giz = mc.iz + gen, *gic = mc.ic + gen;
  const double *ug = mc.ugamma + gen;
  int *noproj = mc.noproj + (size_t)r * nc, *slot = mc.slot + (size_t)r * nc;
  const double *params = mc.params + (size_t)r * nc * np;
  for (int c = warp; c < nc; c += nwarps) {
    const double *z = mc.Z + zidx(mc, giz[c], r, gic[c]) * np;
    const double *cur = params + (size_t)c * np;
    int same = 1;
    for (int p = lane; p < np; p += 32) same &= (z[p] == cur[p]);   // np.all(z == params, axis=1)
    same = __all_sync(0xffffffffu, same) ? 1 : 0;
    if (lane == 0) noproj[c] = same;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int k = mc.usn_off[(size_t)r * (mc.chainsize + 1) + i];
    for (int c = 0; c < nc; c++) if (ug[c] < 0.1 && noproj[c]) slot[c] = k++;
    for (int c = 0; c < nc; c++) if (ug[c] < 0.1 && !noproj[c]) slot[c] = k++;
  }
  __syncthreads();
  const int nfree = mc.nfree;
  for (int c = warp; c < nc; c += nwarps) {
    const size_t g = (size_t)r * nc + c;
    const double *cur = params + (size_t)c * np;
    double *nx = mc.nextp + g * np;
    // i1 / i2 are flat (row, chain) indices of the retrieval's own history (mcmc.py:529-535)
    const double *z1 = mc.Z + zidx(mc, gi1[c] / nc, r, gi1[c] % nc) * np;
    const double *z2 = mc.Z + zidx(mc, gi2[c] / nc, r, gi2[c] % nc) * np;
    const double *z = mc.Z + zidx(mc, giz[c], r, gic[c]) * np;
    const bool sj = ug[c] < 0.1;
    const bool proj = sj && !noproj[c];
    const double *sup = mc.support + (gen + c) * nfree;
    const double *u = sj ? mc.usn + (size_t)slot[c] * nfree : nullptr;
    double dzp = 0.0, d2 = 1.0;
    if (proj) {
      for (int f = lane; f < nfree; f += 32) {
        const int p = mc.ifree[f];
        const double dz = __dsub_rn(cur[p], z[p]);
        s_dz[warp][f] = dz;
        s_t[0][warp][f] = __dmul_rn(z1[p], dz);
        s_t[1][warp][f] = __dmul_rn(z2[p], dz);
        s_t[2][warp][f] = __dmul_rn(dz, dz);
      }
      __syncwarp();
      const double zp1 = np_pairwise_sum(s_t[0][warp], nfree);
      const double zp2 = np_pairwise_sum(s_t[1][warp], nfree);
      d2 = np_pairwise_sum(s_t[2][warp], nfree);
      dzp = __dsub_rn(zp1, zp2);
    }
    int out = 0;
    for (int f = lane; f < nfree; f += 32) {
      const int p = mc.ifree[f];
      double jump;
      if (!sj) jump = __dadd_rn(__dmul_rn(mc.gamma, __dsub_rn(z1[p], z2[p])), __dmul_rn(mc.fepsilon, sup[f]));
      else if (!proj) jump = __dmul_rn(u[f], __dsub_rn(z2[p], z1[p]));
      else jump = __dmul_rn(__ddiv_rn(__dmul_rn(u[f], dzp), d2), s_dz[warp][f]);
      const double lo = mc.pmin[p], hi = mc.pmax[p];
      double v = __dadd_rn(cur[p], jump);
      const int o = (v < lo) || (v > hi);
      out |= o;
      mc.outbounds[g * nfree + f] += o;
      if (v < lo) v = lo;
      if (v > hi) v = hi;
      nx[p] = v;
    }
    out = __any_sync(0xffffffffu, out) ? 1 : 0;
    __syncwarp();                               // the lanes' nx[] are visible to lane 0; s_dz / s_t free again
    if (lane == 0) {
      for (int s = 0; s < mc.nshare; s++) nx[mc.share_dst[s]] = nx[mc.share_src[s]];
      mc.outflag[g] = out;
    }
  }
}

void launch_snooker_propose(const McmcDev &mc, cudaStream_t s) {
  snooker_propose_kernel<<<mc.nretr, kSnkThreads, 0, s>>>(mc);
}

// ---------------------------------------------------------------------------------------
__device__ const double *chain_model(const double *models, const ModelMap &mp, int c, int ndata) {
  // contiguous blocks: the first `extra` ranks own base+1 chains (driver.partition)
  const int cut = mp.extra * (mp.base + 1);
  int r, j;
  if (c < cut) { r = c / (mp.base + 1); j = c - r * (mp.base + 1); }
  else { r = mp.extra + (mp.base > 0 ? (c - cut) / mp.base : 0); j = c - cut - (r - mp.extra) * mp.base; }
  return models + ((size_t)r * mp.pad + j) * ndata;
}

// chisq.c:111-142 + stats.h:72-103: sequential sums; priorup is priorlow at the call sites
// (mcmc.py:338-339,596-597 pass priorlow twice).  data / uncert: the chain's retrieval's.
__device__ __forceinline__ void chain_chisq(const McmcDev &mc, const double *data, const double *uncert,
                                            const double *model, const double *p, double &chisq) {
  double c = 0.0;
  for (int i = 0; i < mc.ndata; i++) {
    const double r = (model[i] - data[i]) / uncert[i];
    c = __dadd_rn(c, __dmul_rn(r, r));
  }
  for (int k = 0; k < mc.nprior; k++) {
    const int ip = mc.iprior[k];
    const double off = p[ip] - mc.prior[ip], lo = mc.priorlow[ip];
    if (lo == -1) c += 2.0 * log(off);
    else { const double r = off / lo; c = __dadd_rn(c, __dmul_rn(r, r)); }
  }
  chisq = c;
}

// chain_chisq by a whole warp: the residuals of 32 data points at a time side by side, their squares
// added in index order (every lane carries the same running sum), priors as in chain_chisq
__device__ __forceinline__ void warp_chain_chisq(const McmcDev &mc, const double *data, const double *uncert,
                                                 const double *model, const double *p, int lane,
                                                 double &chisq, double &c2) {
  double c = 0.0;
  for (int base = 0; base < mc.ndata; base += 32) {
    const int idx = base + lane;
    double r2 = 0.0;
    if (idx < mc.ndata) {
      const double r = (model[idx] - data[idx]) / uncert[idx];
      r2 = __dmul_rn(r, r);
    }
    const int cnt = min(32, mc.ndata - base);
    for (int k = 0; k < cnt; k++) c = __dadd_rn(c, __shfl_sync(0xffffffffu, r2, k));
  }
  double jc = 0.0;
  for (int k = 0; k < mc.nprior; k++) {
    const int ip = mc.iprior[k];
    const double off = p[ip] - mc.prior[ip], lo = mc.priorlow[ip];
    if (lo == -1) { const double t = 2.0 * log(off); c += t; jc += t; }
    else { const double r = off / lo; c = __dadd_rn(c, __dmul_rn(r, r)); }
  }
  chisq = c;
  c2 = c - jc;
}

// first index of the minimum of v[0..n) (np.argmin) by one warp; every lane gets (best, arg)
__device__ __forceinline__ void warp_argmin(const double *v, int n, double &best, int &arg) {
  best = INFINITY;
  arg = 0x7fffffff;
  for (int c = threadIdx.x & 31; c < n; c += 32) {
    const double x = v[c];
    if (x < best || (x == best && c < arg)) { best = x; arg = c; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_down_sync(0xffffffffu, best, o);
    const int oa = __shfl_down_sync(0xffffffffu, arg, o);
    if (ob < best || (ob == best && oa < arg)) { best = ob; arg = oa; }
  }
  best = __shfl_sync(0xffffffffu, best, 0);
  arg = __shfl_sync(0xffffffffu, arg, 0);
}

// One CTA per retrieval; a warp per chain with lanes over the data points / parameters, so that a
// chain's residuals, state copy and trace stores go out side by side (thread-per-chain was ~20
// dependent memory round trips: 11 us at 10 chains).  The snooker norm keeps its 256-slot reduction
// tree.  The CTA advances its retrieval's generation counter (and history size) at the end; no other
// CTA reads them.
constexpr int kChisqThreads = 512;
__global__ void __launch_bounds__(kChisqThreads)
chisq_accept_kernel(McmcDev mc, const double *__restrict__ models, ModelMap mp, int first) {
  const int np = mc.npars, nc = mc.nchains;
  const int r = blockIdx.x;                     // retrieval
  const int g0 = r * nc;                        // its first chain in the flattened population
  const int i = mc.iter[r];
  const bool snooker = mc.walk == 1 && !first;
  const int zrow = snooker ? mc.zsize[r] : 0;
  const size_t gen = ((size_t)r * mc.chainsize + i) * nc;     // generation i of retrieval r in the streams
  const double *data = mc.data + (size_t)r * mc.ndata, *uncert = mc.uncert + (size_t)r * mc.ndata;
  // Metropolis factor of the projected snooker jumps (mcmc.py:603-609): ONE ratio of Frobenius
  // norms over all such chains of this generation, to the power nfree-1 (the reference's
  // np.linalg.norm over the stacked rows; its BLAS summation order is not reproduced, so the
  // factor may differ in the last bit, which only matters for a proposal exactly on the
  // acceptance threshold)
  __shared__ double s_n1[256], s_n2[256];
  double mrf = 1.0;
  if (snooker) {
    if (threadIdx.x < 256) {
      double a1 = 0.0, a2 = 0.0;
      for (int c = threadIdx.x; c < nc; c += 256) {
        const bool sj = mc.ugamma[gen + c] < 0.1;
        if (!sj || mc.noproj[g0 + c] || mc.outflag[g0 + c]) continue;
        const double *z = mc.Z + zidx(mc, mc.iz[gen + c], r, mc.ic[gen + c]) * np;
        const double *cur = mc.params + (size_t)(g0 + c) * np, *nx = mc.nextp + (size_t)(g0 + c) * np;
        for (int f = 0; f < mc.nfree; f++) {
          const int p = mc.ifree[f];
          const double d1 = nx[p] - z[p], d2 = cur[p] - z[p];
          a1 += d1 * d1; a2 += d2 * d2;
        }
      }
      s_n1[threadIdx.x] = a1; s_n2[threadIdx.x] = a2;
    }
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
      if ((int)threadIdx.x < o) { s_n1[threadIdx.x] += s_n1[threadIdx.x + o]; s_n2[threadIdx.x] += s_n2[threadIdx.x + o]; }
      __syncthreads();
    }
    mrf = pow(sqrt(s_n1[0]) / sqrt(s_n2[0]), (double)(mc.nfree - 1));
  }
  const int lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  for (int c = threadIdx.x >> 5; c < nc; c += nwarps) {
    const int g = g0 + c;
    const double *model = chain_model(models, mp, g, mc.ndata);
    double *cur = mc.params + (size_t)g * np;
    if (first) {
      double chisq, c2;
      warp_chain_chisq(mc, data, uncert, model, cur, lane, chisq, c2);
      if (lane == 0) { mc.currchisq[g] = chisq; mc.c2[g] = c2; }
      continue;
    }
    const double *nx = mc.nextp + (size_t)g * np;
    const int oflag = mc.outflag[g];
    const double currc = mc.currchisq[g];
    const double u = mc.unif[gen + c];
    const bool proj = snooker && mc.ugamma[gen + c] < 0.1 && !mc.noproj[g] && !oflag;
    double next = INFINITY, c2 = 0.0;                          // mcmc.py:598
    if (!oflag) warp_chain_chisq(mc, data, uncert, model, nx, lane, next, c2);
    double accept = exp(0.5 * (currc - next));
    if (proj) accept = __dmul_rn(accept, mrf);
    const bool ok = accept >= u;
    const double *state = ok ? nx : cur;                        // the chain's state after this generation
    for (int f = lane; f < mc.nfree; f += 32)
      mc.allparams[((size_t)g * mc.nfree + f) * mc.chainsize + i] = state[mc.ifree[f]];
    if (snooker && (mc.nold + i) % mc.thinning == 0) {         // mcmc.py:653-660
      const size_t zk = zidx(mc, zrow, r, c);
      double *zr = mc.Z + zk * np;
      for (int f = lane; f < mc.nfree; f += 32) zr[mc.ifree[f]] = state[mc.ifree[f]];
      if (lane == 0) mc.Zchisq[zk] = ok ? next : currc;
    }
    {                                                          // mcmc.py:636-651
      double *cm = mc.curmodel + (size_t)g * mc.ndata;
      for (int d = lane; d < mc.ndata; d += 32) {
        const double v = ok ? model[d] : cm[d];
        if (ok) cm[d] = v;
        mc.allmodel[((size_t)g * mc.ndata + d) * mc.chainsize + i] = v;
      }
    }
    __syncwarp();                                              // every lane has read `state` = cur when !ok
    if (ok)
      for (int p = lane; p < np; p += 32) cur[p] = nx[p];
    if (lane == 0) {
      if (!oflag) mc.c2[g] = c2;
      mc.nextchisq[g] = next;
      if (ok) {
        mc.currchisq[g] = next;
        if (mc.nold + i >= mc.burnin) mc.numaccept[g] += 1.0;
      }
    }
  }
  __syncthreads();
  // running best fit: first index of the minimum no-Jeffreys chi-squared (np.argmin)
  if (threadIdx.x < 32) {
    double best;
    int arg;
    warp_argmin(mc.c2 + g0, nc, best, arg);
    const bool take = arg < nc && (first || best < mc.bestchisq[r]);
    if (take) {
      const double *model = chain_model(models, mp, g0 + arg, mc.ndata);
      for (int p = threadIdx.x; p < np; p += 32) mc.bestp[(size_t)r * np + p] = mc.params[(size_t)(g0 + arg) * np + p];
      for (int d = threadIdx.x; d < mc.ndata; d += 32) mc.bestmodel[(size_t)r * mc.ndata + d] = model[d];
    }
    __syncwarp();
    if (threadIdx.x == 0) {
      if (take) mc.bestchisq[r] = best;
      if (!first) mc.iter[r] = i + 1;
      if (snooker && (mc.nold + i) % mc.thinning == 0) mc.zsize[r] = zrow + 1;
    }
  }
}

// chi-squared of the initial Z samples of row `row` and the running best over rows in flattened
// (row, chain) order, first minimum wins like np.argmin (mcmc.py:441-460); Zchisq keeps the value
// WITH the Jeffreys term, which is also what the reference compares to the chains' best (462-470).
// One CTA per retrieval.
__global__ void __launch_bounds__(256)
zrow_chisq_kernel(McmcDev mc, const double *__restrict__ models, ModelMap mp, int row, int last) {
  const int np = mc.npars, nc = mc.nchains, nd = mc.ndata;
  const int r = blockIdx.x, g0 = r * nc;
  const double *data = mc.data + (size_t)r * nd, *uncert = mc.uncert + (size_t)r * nd;
  double *zc = mc.Zchisq + zidx(mc, row, r, 0);
  const double *zs = mc.Z + zidx(mc, row, r, 0) * np;
  double *zbest = mc.zbest + (size_t)r * (1 + np + nd);
  for (int c = threadIdx.x; c < nc; c += blockDim.x)
    chain_chisq(mc, data, uncert, chain_model(models, mp, g0 + c, nd), zs + (size_t)c * np, zc[c]);
  __syncthreads();
  if (threadIdx.x < 32) {
    double best;
    int arg;
    warp_argmin(zc, nc, best, arg);
    const bool take = arg < nc && (row == 0 || best < zbest[0]);
    if (take) {
      const double *model = chain_model(models, mp, g0 + arg, nd);
      for (int p = threadIdx.x; p < np; p += 32) zbest[1 + p] = zs[(size_t)arg * np + p];
      for (int d = threadIdx.x; d < nd; d += 32) zbest[1 + np + d] = model[d];
    }
    __syncwarp();
    if (threadIdx.x == 0 && take) zbest[0] = best;
    __syncwarp();
    if (last && zbest[0] < mc.bestchisq[r]) {
      for (int p = threadIdx.x; p < np; p += 32) mc.bestp[(size_t)r * np + p] = zbest[1 + p];
      for (int d = threadIdx.x; d < nd; d += 32) mc.bestmodel[(size_t)r * nd + d] = zbest[1 + np + d];
      __syncwarp();
      if (threadIdx.x == 0) mc.bestchisq[r] = zbest[0];
    }
  }
}

void launch_zrow_chisq(const McmcDev &mc, const double *models, ModelMap map, int row, int last,
                       cudaStream_t s) {
  zrow_chisq_kernel<<<mc.nretr, 256, 0, s>>>(mc, models, map, row, last);
}

void launch_chisq_accept(const McmcDev &mc, const double *models, ModelMap map, int first,
                         cudaStream_t s) {
  chisq_accept_kernel<<<mc.nretr, kChisqThreads, 0, s>>>(mc, models, map, first);
}

// ---------------------------------------------------------------------------------------
// Random streams of a seeded call (philox.cuh for the generator and the counter layout).  The
// constructions are MC3's (mcmc.py:484-507 for DE-MC, 529-556 for snooker), so the proposal
// distribution is MC3's; only the random numbers differ.

// numpy's legacy polar method (separately rounded, so acceptance decisions are numpy's); a
// rejected pair is followed by the next attempt's
__device__ double polar_normal(unsigned long long k0, unsigned long long k1, long long it, int c, int f) {
  for (int a = 0;; a++) {
    const Philox4 b = draw_block(k0, k1, DRAW_SUPPORT, it, c, f, a);
    const double u = __dsub_rn(__dmul_rn(2.0, u01(b.x[0])), 1.0);
    const double v = __dsub_rn(__dmul_rn(2.0, u01(b.x[1])), 1.0);
    const double s = __dadd_rn(__dmul_rn(u, u), __dmul_rn(v, v));
    if (s > 0.0 && s < 1.0) return __dmul_rn(u, sqrt(__ddiv_rn(__dmul_rn(-2.0, log(s)), s)));
  }
}

// rows of the snooker history at generation i of the call: Z grows after every generation whose
// global iteration is a multiple of the thinning (chisq_accept_kernel)
__device__ __forceinline__ int history_rows(const DrawArgs &d, int i) {
  const long long th = d.thinning, a = d.it0, b = d.it0 + i;
  return d.zs0 + (int)((b + th - 1) / th - (a + th - 1) / th);
}

// one thread per (retrieval, generation, chain): everything but the snooker factor rows
__global__ void __launch_bounds__(256) mcmc_draw_kernel(DrawArgs d) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int nc = d.nchains;
  if (g >= (long long)d.nretr * d.niter * nc) return;
  const int c = (int)(g % nc);
  const long long ri = g / nc;                 // r * niter + i
  const int i = (int)(ri % d.niter), r = (int)(ri / d.niter);
  const unsigned long long k0 = d.keys[2 * r], k1 = d.keys[2 * r + 1];
  const long long it = d.it0 + i;
  for (int f = 0; f < d.nfree; f++)
    d.support[g * d.nfree + f] = __dmul_rn(d.step[f], polar_normal(k0, k1, it, c, f));
  d.unif[g] = u01(draw_block(k0, k1, DRAW_UNIF, it, c, 0, 0).x[0]);
  d.ugamma[g] = u01(draw_block(k0, k1, DRAW_UGAMMA, it, c, 0, 0).x[0]);
  if (d.walk == 0) {                           // mcmc.py:498-505; r1 / r2 are [nretr][nchains][niter]
    int a = randint(draw_block(k0, k1, DRAW_R1, it, c, 0, 0).x[0], 0, nc - 1);
    if (a == c) a = nc - 1;
    int b = (c + randint(draw_block(k0, k1, DRAW_R2, it, c, 0, 0).x[0], 1, nc - 1)) % nc;
    if (b == a) b = (c - 1 + nc) % nc;
    const size_t k = ((size_t)r * nc + c) * d.niter + i;
    d.r1[k] = a;
    d.r2[k] = b;
    return;
  }
  const int zs = history_rows(d, i);           // mcmc.py:529-539
  const long long lim = (long long)(zs - 1) * nc;
  const int a = randint(draw_block(k0, k1, DRAW_I1, it, c, 0, 0).x[0], 0, lim);
  int b, t = 0;
  do b = randint(draw_block(k0, k1, DRAW_I2, it, c, 0, t++).x[0], 0, lim);
  while (b == a);
  d.i1[g] = a;
  d.i2[g] = b;
  d.iz[g] = randint(draw_block(k0, k1, DRAW_IZ, it, c, 0, 0).x[0], 0, zs - 1);
  d.ic[g] = randint(draw_block(k0, k1, DRAW_IC, it, c, 0, 0).x[0], 0, nc);
}

// usn_off[r][i]: first factor row of generation i of retrieval r, rows of the whole call counted
// in (retrieval, generation) order, usn_off[r][niter] = usn_off[r + 1][0].  One CTA: a thread
// counts a contiguous run of generations, the runs' counts are scanned in shared memory.
constexpr int kScanThreads = 1024;
__global__ void __launch_bounds__(kScanThreads) usn_scan_kernel(DrawArgs d) {
  __shared__ int s[kScanThreads];
  const int t = threadIdx.x, nc = d.nchains, n = d.niter;
  const long long E = (long long)d.nretr * n, per = (E + kScanThreads - 1) / kScanThreads;
  const long long lo = min(E, t * per), hi = min(E, lo + per);
  int sum = 0;
  for (long long e = lo; e < hi; e++)
    for (int c = 0; c < nc; c++) sum += d.ugamma[e * nc + c] < 0.1;
  s[t] = sum;
  __syncthreads();
  for (int o = 1; o < kScanThreads; o <<= 1) {
    const int v = t >= o ? s[t - o] : 0;
    __syncthreads();
    s[t] += v;
    __syncthreads();
  }
  int run = s[t] - sum;
  for (long long e = lo; e < hi; e++) {
    const int r = (int)(e / n), i = (int)(e - (long long)r * n);
    d.usn_off[(size_t)r * (n + 1) + i] = run;
    for (int c = 0; c < nc; c++) run += d.ugamma[e * nc + c] < 0.1;
    if (i == n - 1) d.usn_off[(size_t)r * (n + 1) + n] = run;
  }
}

// uniform(1.2, 2.2) factors of the chains with ugamma < 0.1 (mcmc.py:545-556), one row each in chain
// order within a generation; one thread per (retrieval, generation, chain)
__global__ void __launch_bounds__(256) usn_rows_kernel(DrawArgs d) {
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int nc = d.nchains;
  if (g >= (long long)d.nretr * d.niter * nc) return;
  const int c = (int)(g % nc);
  const long long ri = g / nc;
  const int i = (int)(ri % d.niter), r = (int)(ri / d.niter);
  const double *ug = d.ugamma + ri * nc;
  if (!(ug[c] < 0.1)) return;
  int row = d.usn_off[(size_t)r * (d.niter + 1) + i];
  for (int k = 0; k < c; k++) row += ug[k] < 0.1;
  const unsigned long long k0 = d.keys[2 * r], k1 = d.keys[2 * r + 1];
  const double w = 2.2 - 1.2;                  // numpy's uniform(low, high): low + (high - low) u
  for (int f = 0; f < d.nfree; f++)
    d.usn[(size_t)row * d.nfree + f] =
        __dadd_rn(1.2, __dmul_rn(w, u01(draw_block(k0, k1, DRAW_USN, d.it0 + i, c, f, 0).x[0])));
}

void launch_mcmc_draws(const DrawArgs &d, cudaStream_t s) {
  const long long n = (long long)d.nretr * d.niter * d.nchains;
  if (n <= 0) return;
  const int blocks = (int)((n + 255) / 256);
  mcmc_draw_kernel<<<blocks, 256, 0, s>>>(d);
  if (d.walk == 0) return;
  usn_scan_kernel<<<1, kScanThreads, 0, s>>>(d);
  usn_rows_kernel<<<blocks, 256, 0, s>>>(d);
}

// ---------------------------------------------------------------------------------------
// bart_mcmc_retain: a batched strided gather.  Entry k owns blocks [first, first + nblocks) of the
// one launch; a group of `gs` threads (a power of two <= 32) copies one retrieval block
// ("row": outer index o, kept retrieval j) in vectors of `vec` bytes, so the snooker history,
// which is most of the bytes, moves in 16-byte loads and stores.  Integer division happens once
// per row, not per vector.
constexpr int kRetainThreads = 256;
struct RetainJob {
  const void *src;
  void *dst;
  unsigned rows, filled, n_in;             // rows = outer * nkeep; n_in vectors per row
  int vec, gs_log2, first, nblocks;
};
struct RetainLaunch {
  RetainJob j[kMaxRetainCopies];
  int n, nretr, nkeep;
  const int *keep;
};

template <class V>
__device__ __forceinline__ void retain_rows(const RetainJob &c, const RetainLaunch &a) {
  const unsigned gs = 1u << c.gs_log2, lane = threadIdx.x & (gs - 1);
  const unsigned ngroups = (unsigned)c.nblocks * (kRetainThreads >> c.gs_log2);
  const V *src = (const V *)c.src;
  V *dst = (V *)c.dst;
  for (unsigned s = ((blockIdx.x - c.first) * kRetainThreads + threadIdx.x) >> c.gs_log2; s < c.rows;
       s += ngroups) {
    const unsigned o = s / (unsigned)a.nkeep, j = s - o * (unsigned)a.nkeep;
    const V *from = src + ((size_t)min(o, c.filled) * a.nretr + __ldg(a.keep + j)) * c.n_in;
    V *to = dst + (size_t)s * c.n_in;
    for (unsigned e = lane; e < c.n_in; e += gs) to[e] = from[e];
  }
}

__global__ void __launch_bounds__(kRetainThreads) mcmc_retain_kernel(const __grid_constant__ RetainLaunch a) {
  int k = 0;
  while (k + 1 < a.n && (int)blockIdx.x >= a.j[k + 1].first) k++;
  const RetainJob &c = a.j[k];
  if (c.vec == 16) retain_rows<int4>(c, a);
  else if (c.vec == 8) retain_rows<int2>(c, a);
  else retain_rows<int>(c, a);
}

void launch_mcmc_retain(const RetainArgs &a, cudaStream_t s) {
  RetainLaunch L{};
  L.nretr = a.nretr; L.nkeep = a.nkeep; L.keep = a.keep;
  int blocks = 0;
  for (int k = 0; k < a.n; k++) {
    const RetainCopy &c = a.c[k];
    const uintptr_t align = (uintptr_t)c.src | (uintptr_t)c.dst | (uintptr_t)c.inner;
    const int vec = align % 16 == 0 ? 16 : align % 8 == 0 ? 8 : 4;
    RetainJob &j = L.j[L.n];
    j.src = c.src; j.dst = c.dst; j.vec = vec;
    j.rows = (unsigned)(c.outer * a.nkeep);
    j.filled = (unsigned)std::min(c.filled, c.outer - 1);
    j.n_in = (unsigned)(c.inner / vec);
    j.gs_log2 = 0;
    while ((1u << j.gs_log2) < j.n_in && j.gs_log2 < 5) j.gs_log2++;
    const long long threads = (long long)j.rows << j.gs_log2;
    if (threads == 0) continue;
    j.first = blocks;
    j.nblocks = (int)std::min<long long>((threads + kRetainThreads - 1) / kRetainThreads, 148 * 16);
    blocks += j.nblocks;
    L.n++;
  }
  if (!blocks) return;
  mcmc_retain_kernel<<<blocks, kRetainThreads, 0, s>>>(L);
}

}  // namespace bart
