// column_math.cuh -- the arithmetic of the forward model, written once as inline
// host+device functions.  The CUDA kernels in kernels.cu are thin wrappers (thread mapping,
// shared-memory staging) around these; tests/cpu_emu compiles the same functions for the host
// as a TEST-ONLY aid to debug the math without a GPU (the product never runs them on the CPU).
//
// Reference citations are into exosports/BART, modules/transit/{transit,pu}/src.
#pragma once
#include "device.cuh"
#include <cmath>
#include <cstring>
#include <vector>

namespace bart {

constexpr double cPI = 3.141592653589793;
constexpr double cAMU = 1.66053886e-24;
constexpr double cLS = 2.99792458e10;
constexpr double cKB = 1.380658e-16;
constexpr double cH = 6.6260755e-27;
constexpr double cAMAGAT = 2.68678e19;
constexpr double cE0H2 = 4.911e-23;
constexpr double cNAVO = 6.02214076e23;
constexpr double cMICRON = 1e-4;

enum { REJ_TGRID = 1, REJ_TCIA = 2, REJ_SUMQ = 4, REJ_FEWPTS = 8, REJ_NOTOOMUCH = 64 };

// ---------------------------------------------------------------------------------------
// fp64 exp and reciprocal for the column kernels.  libdevice's exp() costs ~45 issue slots per
// call on sm_100 and the column kernels need several per (layer, wavenumber) cell, so the fp64
// pipe (16 lanes per SM sub-partition) is what bounds them.
BART_HD double bits_to_double(long long b) {
#ifdef __CUDA_ARCH__
  return __longlong_as_double(b);
#else
  double d; memcpy(&d, &b, 8); return d;
#endif
}
BART_HD long long double_to_bits(double d) {
#ifdef __CUDA_ARCH__
  return __double_as_longlong(d);
#else
  long long b; memcpy(&b, &d, 8); return b;
#endif
}
BART_HD int hi_word(double d) { return (int)(double_to_bits(d) >> 32); }

// 16-byte pair load (records, pair offsets and grid samples are 16-byte aligned)
struct alignas(16) D2 { double x, y; };
BART_HD D2 ld2(const double *p) { return *reinterpret_cast<const D2 *>(p); }
BART_HD D2 ld2b(const char *p) { return *reinterpret_cast<const D2 *>(p); }
BART_HD double ld1b(const char *p) { return *reinterpret_cast<const double *>(p); }
// Global loads of cell_load: volatile asm, so that they stay where the software pipeline of the
// column kernels puts them (after the consumption of the previous depth's data).
BART_HD D2 ldg2b(const char *p) {
#ifdef __CUDA_ARCH__
  D2 v;
  asm volatile("ld.global.nc.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
  return v;
#else
  return *reinterpret_cast<const D2 *>(p);
#endif
}
BART_HD double ldg1b(const char *p) {
#ifdef __CUDA_ARCH__
  double v;
  asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
#else
  return *reinterpret_cast<const double *>(p);
#endif
}
// 32-byte load of a 4-molecule grid sample: one LDG.256 per lane, so a warp's request is 1 KB of
// contiguous memory (two LDG.128 per lane would each touch every other 16 bytes of that span and
// cost twice the L1 wavefronts).
struct alignas(32) D4 { double x, y, z, w; };
BART_HD D4 ld4b(const char *p) {
#ifdef __CUDA_ARCH__
  D4 v;
  asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];"
               : "=d"(v.x), "=d"(v.y), "=d"(v.z), "=d"(v.w) : "l"(p));
  return v;
#else
  D4 v; memcpy(&v, p, sizeof(v)); return v;
#endif
}

// Warp-uniform decisions of the column kernels.  On the host (tests/cpu_emu, one column at a
// time) they degenerate to the column's own predicate.
#ifdef __CUDA_ARCH__
#define BART_WARP_ALL(p) (__all_sync(0xffffffffu, (p)) != 0)
#define BART_WARP_ANY(p) (__any_sync(0xffffffffu, (p)) != 0)
#else
#define BART_WARP_ALL(p) (p)
#define BART_WARP_ANY(p) (p)
#endif


// exp(x) = 2^n 2^(j/N) e^(r ln2/N) with y = x N/ln2 = (N n + j) + r, |r| <= 1/2, N = 16:
// |r ln2/N| <= 0.0217, so a degree-6 polynomial is exact to 4.5e-16.  The caller supplies y as a
// product a*b (one factor usually a constant that already carries N/ln2), so the reduction is two
// FMAs with the SAME exact product: t = a b + 1.5 2^52 rounds y to the nearest integer m (low
// word of t), r = a b - m is exact.  10 fp64 instructions per exp in all.
// The table (shared memory) holds the bit patterns of 2^(j/N) with (j << 16) subtracted from the
// high word, so that adding (m << 16) -- one integer multiply-add -- yields the high word of
// 2^n 2^(j/N) without masking j out of m.  N = 16 keeps the table inside ONE 128-byte bank row:
// divergent lanes never conflict (the column kernels are bound by shared/L1 wavefronts, not by
// the fp64 pipe; a 128-entry table with a degree-4 polynomial measured slower).
// Arguments must satisfy |x| <= 708 (callers clamp).
constexpr int kExpBits = 4;
constexpr int kExpTabSize = 1 << kExpBits;
constexpr double kExpScale = 23.083120654223414;                 // N / ln2
constexpr double kExpYmax = 700.0 * kExpScale;                   // clamp for y
constexpr double kExpQ1 = 0.04332169878499658;                   // (ln2/N)^k / k!
constexpr double kExpQ2 = 0.0009383847928089872;
constexpr double kExpQ3 = 1.3550807779497457e-05;
constexpr double kExpQ4 = 1.467610032291943e-07;
constexpr double kExpQ5 = 1.2715871950558131e-09;
constexpr double kExpQ6 = 9.181219573844438e-12;

static const unsigned long long kExpTabBits[kExpTabSize] = {
#include "exp_table.inc"
};
// entry j as stored in the kernels' shared-memory table
inline unsigned long long exp_table_entry(int j) {
  return kExpTabBits[j] - ((unsigned long long)j << (32 + 20 - kExpBits));
}
inline void fill_exp_table(unsigned long long *tab) {
  for (int j = 0; j < kExpTabSize; j++) tab[j] = exp_table_entry(j);
}

// exp(a*b*ln2/N) + addend   (addend 0, or -1 for the Planck denominator)
BART_HD double exp_core(double a, double b, const unsigned long long *tab, double addend) {
  const double MAGIC = 6755399441055744.0;                        // 1.5 * 2^52
  const double t = fma(a, b, MAGIC);
  const double kf = t - MAGIC;
  const double r = fma(a, b, -kf);
  double p = kExpQ6;
  p = fma(p, r, kExpQ5);
  p = fma(p, r, kExpQ4);
  p = fma(p, r, kExpQ3);
  p = fma(p, r, kExpQ2);
  p = fma(p, r, kExpQ1);
  p = fma(p, r, 1.0);
#ifdef __CUDA_ARCH__
  const int m = __double2loint(t);
  const uint2 e = *reinterpret_cast<const uint2 *>(tab + (m & (kExpTabSize - 1)));
  const double sc = __hiloint2double((int)(e.y + ((unsigned)m << (20 - kExpBits))), (int)e.x);
#else
  const int m = (int)double_to_bits(t);
  const unsigned long long e = tab[m & (kExpTabSize - 1)];
  const unsigned hi = (unsigned)(e >> 32) + ((unsigned)m << (20 - kExpBits));
  const double sc = bits_to_double((long long)(((unsigned long long)hi << 32) | (e & 0xffffffffull)));
#endif
  return fma(p, sc, addend);
}
// exp(x) for x <= 0, any magnitude (0 below -700 up to 1e-304: the argument is clamped)
BART_HD double fast_exp_neg(double x, const unsigned long long *tab) {
  return exp_core(x < -700.0 ? -700.0 : x, kExpScale, tab, 0.0);
}
// exp(x), saturating: |x| clamped to 700
BART_HD double fast_exp(double x, const unsigned long long *tab) {
  x = x < -700.0 ? -700.0 : x;
  x = x > 700.0 ? 700.0 : x;
  return exp_core(x, kExpScale, tab, 0.0);
}

// Reduced-degree variants for the eclipse column kernel, whose instruction count is what bounds it
// (DESIGN.md section 4).  Coefficients interpolate e^(r ln2/N) at the Chebyshev nodes of
// |r| <= 1/2: degree 4 is within 2.6e-12 relative, degree 5 within 9e-15 (tests/test_emu_math.py).
constexpr double kExp4C1 = 0.043321698760160544, kExp4C2 = 0.0009383847926296646,
                 kExp4C3 = 1.3551205154935067e-05, kExp4C4 = 1.4676387238435006e-07;
constexpr double kExp5C1 = 0.04332169878499661, kExp5C2 = 0.000938384792486206,
                 kExp5C3 = 1.355080777749983e-05, kExp5C4 = 1.467644462189871e-07,
                 kExp5C5 = 1.2716085030349987e-09;
constexpr double kExpMagic = 6755399441055744.0;                  // 1.5 * 2^52

// table value for the low word m of the rounded sum t: 2^(m/N) (or wgt 2^(m/N) from an angle's
// table) -- layout: exp_table_entry
BART_HD double exp_scale(double t, const unsigned long long *tab) {
#ifdef __CUDA_ARCH__
  const int m = __double2loint(t);
  const uint2 e = *reinterpret_cast<const uint2 *>(tab + (m & (kExpTabSize - 1)));
  return __hiloint2double((int)(e.y + ((unsigned)m << (20 - kExpBits))), (int)e.x);
#else
  const int m = (int)double_to_bits(t);
  const unsigned long long e = tab[m & (kExpTabSize - 1)];
  const unsigned hi = (unsigned)(e >> 32) + ((unsigned)m << (20 - kExpBits));
  return bits_to_double((long long)(((unsigned long long)hi << 32) | (e & 0xffffffffull)));
#endif
}
// exp(a*b*ln2/N) + addend, degree 5
BART_HD double exp_core5(double a, double b, const unsigned long long *tab, double addend) {
  const double t = fma(a, b, kExpMagic);
  const double r = fma(a, b, -(t - kExpMagic));
  double p = kExp5C5;
  p = fma(p, r, kExp5C4);
  p = fma(p, r, kExp5C3);
  p = fma(p, r, kExp5C2);
  p = fma(p, r, kExp5C1);
  p = fma(p, r, 1.0);
  return fma(p, exp_scale(t, tab), addend);
}
// acc + s exp(a*b*ln2/N), degree 4, 8 fp64 instructions; s is whatever factor `tab` carries (1 for
// the plain table, the angle's weight for its own table: fill_ecl_exp_table)
BART_HD double exp_w(double a, double b, const unsigned long long *tab, double acc) {
  const double t = fma(a, b, kExpMagic);
  const double r = fma(a, b, -(t - kExpMagic));
  double p = kExp4C4;
  p = fma(p, r, kExp4C3);
  p = fma(p, r, kExp4C2);
  p = fma(p, r, kExp4C1);
  p = fma(p, r, 1.0);
  return fma(p, exp_scale(t, tab), acc);
}

// 1/d for finite d > 0 to 2^-44: hardware seed (MUFU.RCP64H, 2^-22) + one Newton step
BART_HD double fast_rcp1(double d) {
#ifdef __CUDA_ARCH__
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
  const double e = fma(-d, r, 1.0);
  return fma(r, e, r);
#else
  return 1.0 / d;
#endif
}

// 1/d for finite d > 0: hardware seed (MUFU.RCP64H) + two Newton steps; the compiler's IEEE
// divide is ~3x the issue slots because of its special-case branches.
BART_HD double fast_rcp(double d) {
#ifdef __CUDA_ARCH__
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
  double e = fma(-d, r, 1.0);      // seed: >= 20 bits
  r = fma(r, e, r);                // 2^-40
  e = fma(-d, r, 1.0);
  r = fma(r, e, r);                // below rounding
  return r;
#else
  return 1.0 / d;
#endif
}

// Angle constants of the eclipse geometry (filled on the host at init):
//   D(tau) = sum_a wgt[a] exp(-tau inv_mu[a]), the hemispheric transmission that weights the
//   Planck function (eclipse_intens + flux, eclipse.c:117-160,242-287, are linear in the
//   per-angle intensities, so the angle sum can be taken before the layer integral).
//   For tau <= tau_small D is one polynomial of degree kTaylorN - 1 in u = 2 tau / tau_small - 1: the
//   Chebyshev interpolant of D on [0, tau_small], converted to the monomial basis in long double.
//   At the same degree it reaches four times further than the Maclaurin series it replaced
//   (tau max(inv_mu) <= 2 instead of 0.5 at 5e-13), which moves ~10 % of the (slot, depth) steps
//   from the weighted exponentials to 13 instructions: eclipse kernel 4.30 -> 4.11 ms.
inline void fill_angle_consts(DevConfig &c) {
  double smax = 0.0;
  for (int a = 0; a < c.nang; a++) {
    c.exp_a[a] = c.inv_mu[a] * kExpScale;
    if (c.inv_mu[a] > smax) smax = c.inv_mu[a];
  }
  double d0 = 0.0;                                           // sequential sum, like the angle loop
  for (int a = 0; a < c.nang; a++) d0 = fma(1.0, c.wgt[a], d0);
  c.d0 = d0;
  auto Dref = [&](long double tau) {
    long double acc = 0.0L;
    for (int a = 0; a < c.nang; a++) acc += (long double)c.wgt[a] * expl(-tau * (long double)c.inv_mu[a]);
    return acc;
  };
  // range: tau max(inv_mu) <= 2, halved until the interpolant is within 2e-12 D(0) of the sum
  double reach = 2.0;
  for (int attempt = 0; attempt < 8; attempt++, reach *= 0.5) {
    c.tau_small = smax > 0 ? reach / smax : 0.0;
    c.ser_s = c.tau_small > 0 ? 2.0 / c.tau_small : 0.0;
    const long double half = (long double)c.tau_small / 2, pi = 3.14159265358979323846264338327950288L;
    long double f[kTaylorN], cheb[kTaylorN];
    for (int j = 0; j < kTaylorN; j++) f[j] = Dref(half + half * cosl(pi * (j + 0.5L) / kTaylorN));
    for (int k = 0; k < kTaylorN; k++) {
      long double acc = 0.0L;
      for (int j = 0; j < kTaylorN; j++) acc += f[j] * cosl(pi * k * (j + 0.5L) / kTaylorN);
      cheb[k] = acc * 2.0L / kTaylorN;
    }
    cheb[0] /= 2;
    long double t0[kTaylorN] = {0}, t1[kTaylorN] = {0}, t2[kTaylorN], mono[kTaylorN] = {0};
    t0[0] = 1.0L; t1[1] = 1.0L;                              // T_0, T_1 in powers of u
    for (int k = 0; k < kTaylorN; k++) {
      const long double *tk = k == 0 ? t0 : t1;
      if (k >= 2) {                                          // T_k = 2 u T_{k-1} - T_{k-2}
        for (int i = 0; i < kTaylorN; i++) t2[i] = (i > 0 ? 2 * t1[i - 1] : 0.0L) - t0[i];
        for (int i = 0; i < kTaylorN; i++) { t0[i] = t1[i]; t1[i] = t2[i]; }
        tk = t1;
      }
      for (int i = 0; i < kTaylorN; i++) mono[i] += cheb[k] * tk[i];
    }
    for (int i = 0; i < kTaylorN; i++) c.taylor[i] = (double)mono[i];
    double worst = 0.0;
    for (int t = 0; t <= 2000; t++) {
      const double tau = c.tau_small * t / 2000.0;
      const double u = fma(tau, c.ser_s, -1.0);
      double p = c.taylor[kTaylorN - 1];
      for (int i = kTaylorN - 2; i >= 0; i--) p = fma(p, u, c.taylor[i]);
      worst = fmax(worst, fabs(p - (double)Dref(tau)));
    }
    if (worst <= 2e-12 * fabs(d0) || c.tau_small == 0.0) break;
  }
  c.sq_src = c.sq_dst = -1;
  for (int b = 0; b < c.nang && c.sq_dst < 0; b++)
    for (int a = 0; a < b; a++)
      if (fabs(c.inv_mu[b] - 2.0 * c.inv_mu[a]) <= 4e-16 * c.inv_mu[b] && fabs(c.wgt[a]) > 1e-100) {
        c.sq_src = a; c.sq_dst = b; break;
      }
  // the clamp keeps wgt exp(-tau inv_mu) a normal number (the weights live in the angle tables)
  double lnw_min = 0.0;
  for (int a = 0; a < c.nang; a++)
    if (fabs(c.wgt[a]) > 1e-100 && log(fabs(c.wgt[a])) < lnw_min) lnw_min = log(fabs(c.wgt[a]));
  c.tau_clamp = (690.0 + lnw_min) / (smax > 0 ? smax : 1.0);
  c.sq_coef = c.sq_dst >= 0 ? c.wgt[c.sq_dst] / (c.wgt[c.sq_src] * c.wgt[c.sq_src]) : 0.0;
}

// Shared-memory exp tables of the eclipse kernel: the plain 2^(j/N) table followed by one table per
// ray angle holding wgt[a] 2^(j/N) (same biased layout), kEclTabEntries(nang) entries in all.  A
// weight below 1e-100 in magnitude counts as zero: its table holds 2^-1000 2^(j/N).
BART_HD int ecl_tab_entries(int nang) { return (1 + nang) * kExpTabSize; }
inline void fill_ecl_exp_table(const DevConfig &c, unsigned long long *tab) {
  fill_exp_table(tab);
  for (int a = 0; a < c.nang; a++) {
    const long double w = fabs(c.wgt[a]) > 1e-100 ? (long double)c.wgt[a] : ldexpl(1.0L, -1000);
    for (int j = 0; j < kExpTabSize; j++) {
      const double v = (double)(w * exp2l((long double)j / kExpTabSize));
      tab[(1 + a) * kExpTabSize + j] =
          (unsigned long long)double_to_bits(v) - ((unsigned long long)j << (32 + 20 - kExpBits));
    }
  }
}

// CIA tables for the device: [T_k][wave][4] = (P_k, Q_k, P_k+1, Q_k+1) (P = table column splined
// onto the spectrum grid, Q = its temperature second derivative; the last node repeats itself),
// followed by `pad` samples of zeros.
inline std::vector<double> pack_cia_quads(const std::vector<double> &P, const std::vector<double> &Q,
                                          int nt, int nw, int pad) {
  std::vector<double> out((size_t)nt * nw * 4 + (size_t)pad * 4, 0.0);
  for (int k = 0; k < nt; k++) {
    const int k1 = k + 1 < nt ? k + 1 : k;
    for (int w = 0; w < nw; w++) {
      double *o = &out[((size_t)k * nw + w) * 4];
      o[0] = P[(size_t)k * nw + w];  o[1] = Q[(size_t)k * nw + w];
      o[2] = P[(size_t)k1 * nw + w]; o[3] = Q[(size_t)k1 * nw + w];
    }
  }
  return out;
}

struct KnobVals {
  double r0;
  int cloud_flag; double cloudext, cloudtop, cloudbot;
  int scat_flag; double scat_logext;
};

BART_HD KnobVals knobs_for(const Knobs &k, int m) {
  KnobVals v;
  v.r0 = k.r0 ? k.r0[m] : k.r0_all;
  if (k.cloudtop) {                       // set_cloudtop semantics, transit.c:103-109
    v.cloud_flag = 1; v.cloudext = 100.0; v.cloudtop = k.cloudtop[m]; v.cloudbot = k.cloudtop[m] + 10;
  } else {
    v.cloud_flag = k.cloud_flag_all; v.cloudext = k.cloudext_all;
    v.cloudtop = k.cloudtop_all; v.cloudbot = k.cloudbot_all;
  }
  v.scat_flag = k.scat_flag ? k.scat_flag[m] : k.scat_flag_all;
  v.scat_logext = k.scat_logext ? k.scat_logext[m] : k.scat_logext_all;
  return v;
}

// ---------------------------------------------------------------------------------------
// The configuration arrays the preparation stages read, by pointer: atm_prep_kernel points them at
// its shared-memory copies (the kernel parameter itself stays read-only), everything else at the
// configuration's own arrays (prep_ptrs_of).
struct PrepPtrs {
  const double *press, *gtemp, *mass, *pol;
  const double *ciaT[kMaxCia];
};
BART_HD PrepPtrs prep_ptrs_of(const DevConfig &c) {
  PrepPtrs q;
  q.press = c.press; q.gtemp = c.gtemp; q.mass = c.mass; q.pol = c.pol;
  for (int f = 0; f < kMaxCia; f++) q.ciaT[f] = c.ciaT[f];
  return q;
}

// atm_prep stage 1, one layer: mean molecular mass and mass densities.
// Reference: checkaddmm readatm.c:122-159 (number abundances), stateeqnford transit.h:58-69,
// reloadatm readatm.c:722-784.  rho[j*rho_stride] receives the density of species j.
// mass density of species j at layer l
BART_HD double prep_density(const DevConfig &c, const PrepPtrs &pp, const double *in, int l, int j) {
  const double T = in[l];
  const double p = pp.press[l] * c.pfct;
  const double q = in[(size_t)c.nlayer * (j + 1) + l];
  const double r = cAMU * q * p / cKB / T;
  return r * pp.mass[j];
}
// mean molecular mass of layer l (species in file order) and the abundance-sum test
BART_HD int prep_mu(const DevConfig &c, const PrepPtrs &pp, const double *in, int l, double *mu_out) {
  double mu = 0.0, sumq = 0.0;
  for (int j = 0; j < c.nspec; j++) {
    const double q = in[(size_t)c.nlayer * (j + 1) + l];
    mu += q * pp.mass[j];
    sumq += q;
  }
  *mu_out = mu;
  return sumq > 1.001 ? REJ_SUMQ : 0;
}
BART_HD int prep_layer(const DevConfig &c, const PrepPtrs &pp, const double *in, int l,
                       double *rho, int rho_stride, double *mu_out) {
  for (int j = 0; j < c.nspec; j++) rho[(size_t)j * rho_stride] = prep_density(c, pp, in, l, j);
  return prep_mu(c, pp, in, l, mu_out);
}
BART_HD int prep_layer(const DevConfig &c, const double *in, int l, double *rho, int rho_stride,
                       double *mu_out) {
  return prep_layer(c, prep_ptrs_of(c), in, l, rho, rho_stride, mu_out);
}

// atm_prep stage 2: hydrostatic radii.  Reference: radpress readatm.c:787-865 integrates
//   r_i = r_{i+1} - 1/2 (T_i/mu_i + T_{i+1}/mu_{i+1}) (KB/AMU ln(p_i/p_{i+1}) / g_{i+1}) / rfct
// with the gravity carried along as g <- g (r_{i+1}/r_i)^2, i.e. g_i = g0 (r0/r_i)^2.  Here the
// layer-only factor hc_i = 1/2 (T_i/mu_i + T_{i+1}/mu_{i+1}) KB/AMU ln(p_i/p_{i+1}) / rfct is
// computed in parallel over layers (hydro_coef) and the sequential part is the two-instruction
// recurrence r_i = r_{i+1} - hc_i r_{i+1}^2 / (g0 r0^2) (hydrostatic_radii); the gravity product
// telescopes, so the results agree with the reference's running product to rounding (1e-15).
BART_HD double hydro_coef(const DevConfig &c, const PrepPtrs &pp, const double *temp, const double *mu, int i) {
  return 0.5 * (temp[i] / mu[i] + temp[i + 1] / mu[i + 1]) *
         (cKB / cAMU * log(pp.press[i] / pp.press[i + 1])) / c.rfct;
}
BART_HD double hydro_coef(const DevConfig &c, const double *temp, const double *mu, int i) {
  return hydro_coef(c, prep_ptrs_of(c), temp, mu, i);
}

// the layer nearest to the reference pressure p0 (first minimum of |p - p0|, radpress
// readatm.c:809-813): a property of the configuration, found once on the host
inline int ref_layer_of(const double *press, int nl, double p0) {
  int i0 = 0;
  double best = 1e37;
  for (int i = 0; i < nl; i++) {
    const double d = fabs(press[i] - p0);
    if (d < best) { i0 = i; best = d; }
  }
  return i0;
}

// dirs: bit 0 = walk the layers below the reference layer, bit 1 = those above; either walk
// computes the reference layer's radius itself, so two threads can take one direction each.  The
// coefficient of the next step is fetched before the current step's radius is stored (the
// recurrence is the kernel's longest dependent chain at small batches).
BART_HD void hydrostatic_radii(const DevConfig &c, const PrepPtrs &pp, double r0, const double *temp,
                               const double *mu, const double *hc, double *radius, int dirs = 3) {
  const int nl = c.nlayer;
  const double *pr = pp.press;
  const double p0 = c.p0, g0 = c.gsurf, rfct = c.rfct;
  const int i0 = c.ref_layer;                 // nearest layer to the reference pressure (ref_layer_of)
  if (pr[i0] > p0) {
    const int i1 = i0 + 1 < nl ? i0 + 1 : i0;
    const double lr = log(pr[i1] / pr[i0]), lp = log(p0 / pr[i0]);
    const double t0 = temp[i0] + ((temp[i1] - temp[i0]) / lr) * lp;
    const double m0 = mu[i0] + ((mu[i1] - mu[i0]) / lr) * lp;
    radius[i0] = r0 + 0.5 * (temp[i0] / mu[i0] + t0 / m0) * (cKB / cAMU * lp / g0) / rfct;
  } else {
    const int i1 = i0 > 0 ? i0 - 1 : i0;
    const double lr = log(pr[i1] / pr[i0]), lp = log(p0 / pr[i0]);
    const double t0 = temp[i0] + ((temp[i1] - temp[i0]) / lr) * lp;
    const double m0 = mu[i0] + ((mu[i1] - mu[i0]) / lr) * lp;
    radius[i0] = r0 - 0.5 * (temp[i0] / mu[i0] + t0 / m0) * (cKB / cAMU * log(pr[i0] / p0) / g0) / rfct;
  }
  const double q = 1.0 / (g0 * r0 * r0);
  const double ri0 = radius[i0];
  if ((dirs & 1) && i0 > 0) {
    double r = ri0, h = hc[i0 - 1] * q;
    for (int i = i0 - 1; i >= 0; i--) {
      const double hn = i > 0 ? hc[i - 1] * q : 0.0;
      r = fma(-h, r * r, r);
      radius[i] = r;
      h = hn;
    }
  }
  if ((dirs & 2) && i0 + 1 < nl) {
    double r = ri0, h = hc[i0] * q;
    for (int i = i0 + 1; i < nl; i++) {
      const double hn = i + 1 < nl ? hc[i] * q : 0.0;
      r = fma(h, r * r, r);
      radius[i] = r;
      h = hn;
    }
  }
}

BART_HD void hydrostatic_radii(const DevConfig &c, double r0, const double *temp, const double *mu,
                               const double *hc, double *radius) {
  hydrostatic_radii(c, prep_ptrs_of(c), r0, temp, mu, hc, radius);
}

// floor-bracket search: the reference finds the NEAREST node (iomisc.c:1088-1108) and steps
// down when the value is below it (extinction.c:560-564, spline.c:149-154), i.e. the largest k
// with x[k] <= v, clamped so that k+1 is a valid node.
BART_HD int bracket(const double *x, int n, double v) {
  int lo = 0, hi = n - 1;
  while (hi - lo > 1) {
    const int mid = (hi + lo) >> 1;
    if (x[mid] > v) hi = mid; else lo = mid;
  }
  if (lo > n - 2) lo = n - 2;
  if (lo < 0) lo = 0;
  return lo;
}

// atm_prep stage 3, one depth d (0 = top): every per-layer coefficient the column kernels need,
// written as one record (layout: TabLayout).  temp/radius are indexed by layer (bottom -> top);
// rho[j*rho_stride + layer].
// The record of depth d in four independent parts (disjoint fields), so that atm_prep_kernel can
// deal them to different threads: thermal (temperature, Planck chaining factor, opacity-grid
// bracket and weights), CIA, scattering / cloud, and the radius-dependent quadrature coefficients.
BART_HD int prep_row_thermal(const DevConfig &c, const PrepPtrs &pp, int d, const double *temp,
                             const double *rho, int rho_stride, double *tab, int model = 0) {
  const TabLayout &L = c.lay;
  const int nl = c.nlayer;
  const int l = nl - 1 - d;
  const double T = temp[l];
  double *row = tab + (size_t)d * L.nf();
  int status = 0;
  row[L.T] = T;
  row[L.INVT] = 1.0 / T;
  row[L.PF] = c.planck_cols > 0 ? exp(c.planck_step / T) : 1.0;
  row[L.GOFF + 1] = 0.0;

  // opacity-grid bracket and folded weights (interpolmolext, extinction.c:534-581)
  if (T < pp.gtemp[0] || T > pp.gtemp[c.ntemp - 1]) status |= REJ_TGRID;
  const int it = bracket(pp.gtemp, c.ntemp, T);
  const double t0 = pp.gtemp[it], t1 = pp.gtemp[it + 1];
  row[L.GOFF] = bits_to_double((((long long)l * c.ntemp + it) * c.gms) * (long long)c.nwave * 8);
  if (c.lbl) {
    // line-by-line mode: the "grid" is ext[model][layer][wave] with the densities folded in
    // (computemolext permol = 0, extinction.c:472-473); gtemp = TLI range (makesample.c:488-503)
    row[L.GOFF] = bits_to_double(((long long)model * nl + l) * (long long)c.nwave * 8);
    row[L.W] = 1.0;
    row[L.W + 1] = 0.0;
  }
  for (int m = 0; m < (c.lbl ? 0 : c.ngmol); m++) {
    const double r = rho[(size_t)c.gmol_spec[m] * rho_stride + l];
    row[L.W + 2 * m] = r * (t1 - T) / (t1 - t0);
    row[L.W + 2 * m + 1] = r * (T - t0) / (t1 - t0);
  }
  return status;
}

// CIA: cubic-spline-in-T coefficients (splinterp_pt, spline.c:131-183) applied to the
// wavenumber-pre-splined tables, times the density product (interpcs, crosssec.c:321-336)
BART_HD int prep_row_cia(const DevConfig &c, const PrepPtrs &pp, int d, const double *temp,
                         const double *rho, int rho_stride, double *tab) {
  const TabLayout &L = c.lay;
  const int l = c.nlayer - 1 - d;
  const double T = temp[l];
  double *row = tab + (size_t)d * L.nf();
  int status = 0;
#pragma unroll
  for (int f = 0; f < kMaxCia; f++) {
    if (f >= c.ncia) break;
    const double *x = pp.ciaT[f];
    const int nt = c.cia_nt[f];
    if (T < x[0] || T > x[nt - 1]) status |= REJ_TCIA;
    const int k = bracket(x, nt, T);
    double dens = 1.0;
    for (int s = 0; s < c.cia_nspec[f]; s++) {
      const int sp = c.cia_spec[f][s];
      dens *= rho[(size_t)sp * rho_stride + l] / (cAMU * pp.mass[sp] * cAMAGAT);
    }
    double cy0, cy1, cz0, cz1;
    if (x[k] == T) { cy0 = 1.0; cy1 = 0.0; cz0 = 0.0; cz1 = 0.0; }
    else {
      const double h = x[k + 1] - x[k], dx = T - x[k];
      const double u = dx / h;
      cy0 = 1.0 - u;
      cy1 = u;
      cz0 = dx * (-h / 3.0 + dx * (0.5 - dx / (6.0 * h)));
      cz1 = dx * (-h / 6.0 + dx * dx / (6.0 * h));
    }
    double *cr = row + L.cia(f);
    cr[0] = bits_to_double((long long)k * c.nwave * 32);
    cr[1] = (double)k;
    cr[2] = cy0 * dens;
    cr[3] = cy1 * dens;
    cr[4] = cz0 * dens;
    cr[5] = cz1 * dens;
  }
  return status;
}

BART_HD void prep_row_scat(const DevConfig &c, const PrepPtrs &pp, const KnobVals &kv, int d,
                           const double *temp, const double *rho, int rho_stride, double *tab) {
  const TabLayout &L = c.lay;
  const int l = c.nlayer - 1 - d;
  const double T = temp[l];
  double *row = tab + (size_t)d * L.nf();
  // scattering (computeextscat, extinction.c:586-624): coefficient of wn^4
  double sc = 0.0;
  if (kv.scat_flag == 1) sc = pow(10.0, kv.scat_logext) * cE0H2 * pp.press[l] / T;
  else if (kv.scat_flag == 2) {
    const double k4 = (2.0 * cPI * cMICRON) * (2.0 * cPI * cMICRON) * (2.0 * cPI * cMICRON) *
                      (2.0 * cPI * cMICRON);
    for (int j = 0; j < c.nspec; j++)
      sc += cPI * 8e-32 / 3.0 * (pp.pol[j] * pp.pol[j]) * k4 * rho[(size_t)j * rho_stride + l] /
            pp.mass[j] * cNAVO;
  }
  row[L.SCAT] = sc;

  // gray cloud deck (computeextcloud flag 1, extinction.c:629-693)
  double cl = 0.0;
  if (kv.cloud_flag == 1 && kv.cloudext != 0.0) {
    const double top = pow(10.0, kv.cloudtop), bot = pow(10.0, kv.cloudbot);
    if (pp.press[l] >= top && pp.press[l] < bot) cl = kv.cloudext;
  }
  row[L.CLOUD] = cl;
}

// Simpson / trapezoid coefficients on the radius spacing (geth + simpson, numerical.c:390-525),
// top-aligned panels: the panel ending at even depth d spans depths d-2, d-1, d.
BART_HD void prep_row_radius(const DevConfig &c, int d, const double *radius, double *tab) {
  const TabLayout &L = c.lay;
  const int l = c.nlayer - 1 - d;
  double *row = tab + (size_t)d * L.nf();
  row[L.RAD] = radius[l];
  double sa = 0.0, sb = 0.0, scf = 0.0, tr = 0.0;
  if (d >= 1) {
    const double h0 = radius[l + 1] - radius[l];            // interval (d, d-1)
    tr = c.rfct * h0 / 2.0;
    if (d >= 2) {
      const double h1 = radius[l + 2] - radius[l + 1];      // interval (d-1, d-2)
      const double hsum = h0 + h1, hratio = h1 / h0, hfactor = hsum * hsum / (h0 * h1);
      const double s6 = c.rfct * hsum / 6.0;
      sa = (2.0 - hratio) * s6;
      sb = hfactor * s6;
      scf = (2.0 - 1.0 / hratio) * s6;
    }
  }
  row[L.SA] = sa;
  row[L.SB] = sb;
  row[L.SC] = scf;
  row[L.TR] = tr;
}

BART_HD int prep_table_row(const DevConfig &c, const PrepPtrs &pp, const KnobVals &kv, int d,
                           const double *temp, const double *rho, int rho_stride, const double *radius,
                           double *tab, int model = 0) {
  int status = prep_row_thermal(c, pp, d, temp, rho, rho_stride, tab, model);
  status |= prep_row_cia(c, pp, d, temp, rho, rho_stride, tab);
  prep_row_scat(c, pp, kv, d, temp, rho, rho_stride, tab);
  prep_row_radius(c, d, radius, tab);
  return status;
}
BART_HD int prep_table_row(const DevConfig &c, const KnobVals &kv, int d, const double *temp,
                           const double *rho, int rho_stride, const double *radius, double *tab,
                           int model = 0) {
  return prep_table_row(c, prep_ptrs_of(c), kv, d, temp, rho, rho_stride, radius, tab, model);
}

// ---------------------------------------------------------------------------------------
// Per-column base addresses into the grid and the CIA tables (byte pointers: the table records
// carry byte offsets, so a cell address is one 64-bit add).
struct ColPtrs {
  const char *g;
  const char *cia[kMaxCia];
};
template <int NCIA>
BART_HD ColPtrs col_ptrs(const DevConfig &c, int w) {
  ColPtrs P;
  P.g = reinterpret_cast<const char *>(c.grid) + (size_t)w * c.gms * 8;
#pragma unroll
  for (int f = 0; f < (NCIA >= 0 ? NCIA : kMaxCia); f++)
    P.cia[f] = f < c.ncia ? reinterpret_cast<const char *>(c.ciaPQ[f]) + (size_t)w * 32 : nullptr;
  return P;
}

// Total extinction of one (depth, wavenumber) cell: opacity-grid lookup with temperature
// interpolation and abundance scaling (extinction.c:534-581), + scattering + cloud + CIA in the
// reference's summation order (tau.c:231-232).  `row` is the depth's table record.  NMOL / NCIA
// are compile-time counts (NMOL 0 / NCIA -1 = take them from the configuration at run time).
// The lookup is split into cell_load (issues the global loads: one 8/16/32-byte vector per
// bracketing temperature plane carrying all molecules of the sample, one 32-byte vector per CIA
// file carrying both temperature nodes) and cell_combine (the arithmetic), so that a column kernel
// can issue the loads of the next depth before it works on the current one.
template <int NMOL, int NCIA>
struct CellData {
  static constexpr bool kStatic = NMOL >= 1 && NMOL <= 4;      // grid sample preloaded (vector load)
  static constexpr bool kStaticCia = kStatic && NCIA >= 0;     // CIA samples preloaded too
  static constexpr int NG = !kStatic ? 1 : (NMOL == 1 ? 1 : (NMOL == 2 ? 2 : 4));
  static constexpr int NC = kStaticCia && NCIA > 0 ? NCIA : 1;
  double lo[NG], hi[NG];
  D4 q[NC];                                                    // (P_k, Q_k, P_k+1, Q_k+1)
};

// Byte offsets of one depth's samples from the column pointers: grid plane (layer, it) and the CIA
// bracket rows, as stored in the table record.
template <int NCIA>
struct CellOffs {
  long long g;
  long long cia[NCIA > 0 ? NCIA : 1];
};
template <int NMOL, int NCIA>
BART_HD CellOffs<NCIA> cell_offsets(const double *row) {
  typedef TabLayout L;
  CellOffs<NCIA> o;
  o.g = double_to_bits(row[L::GOFF]);
#pragma unroll
  for (int f = 0; f < (NCIA > 0 ? NCIA : 0); f++) o.cia[f] = double_to_bits(row[L::W + 2 * NMOL + 6 * f]);
  return o;
}

// goff / coff: byte offsets of this column from the column P addresses (grid / CIA tables); as
// compile-time constants they become the immediate offsets of the load instructions
// with_cia false: only the grid samples are loaded and x.q keeps what it holds (a caller that
// walks down a column reloads the CIA samples only when the layer's bracket row changes)
template <int NMOL, int NCIA>
BART_HD void cell_load_at(const DevConfig &c, const ColPtrs &P, const CellOffs<NCIA> &o,
                          CellData<NMOL, NCIA> &x, size_t goff = 0, size_t coff = 0,
                          bool with_cia = true) {
  if (!CellData<NMOL, NCIA>::kStatic) return;                  // run-time counts: loaded in cell_combine
  const size_t plane = (size_t)c.nwave * c.gms * 8;
  const char *lo = P.g + o.g;
  const char *hi = lo + plane;
  if (NMOL == 1) { x.lo[0] = ldg1b(lo + goff); x.hi[0] = ldg1b(hi + goff); }
  else if (NMOL == 2) {
    const D2 a = ldg2b(lo + goff), b = ldg2b(hi + goff);
    x.lo[0] = a.x; x.lo[1] = a.y; x.hi[0] = b.x; x.hi[1] = b.y;
  } else {
    const D4 a = ld4b(lo + goff), b = ld4b(hi + goff);
    x.lo[0] = a.x; x.lo[1] = a.y; x.lo[2] = a.z; x.lo[3] = a.w;
    x.hi[0] = b.x; x.hi[1] = b.y; x.hi[2] = b.z; x.hi[3] = b.w;
  }
  if (!CellData<NMOL, NCIA>::kStaticCia || !with_cia) return;
#pragma unroll
  for (int f = 0; f < (NCIA > 0 ? NCIA : 0); f++) x.q[f] = ld4b(P.cia[f] + o.cia[f] + coff);
}

template <int NMOL, int NCIA>
BART_HD void cell_load(const DevConfig &c, const ColPtrs &P, const double *row,
                       CellData<NMOL, NCIA> &x, size_t goff = 0, size_t coff = 0) {
  if (!CellData<NMOL, NCIA>::kStatic) return;
  cell_load_at<NMOL, NCIA>(c, P, cell_offsets<NMOL, NCIA>(row), x, goff, coff);
}

template <int NMOL, int NCIA, bool SC = true>
BART_HD double cell_combine(const DevConfig &c, const ColPtrs &P, const double *row,
                            const CellData<NMOL, NCIA> &x, double wn4, int part,
                            size_t goff = 0, size_t coff = 0) {
  // part: 0 = total extinction, 1 = molecular lines only, 2 = collision-induced absorption only
  // SC false: the caller knows that the scattering and cloud terms of every record are zero
  typedef TabLayout L;
  const int ngmol = NMOL > 0 ? NMOL : c.ngmol;
  const int ncia = NCIA >= 0 ? NCIA : c.ncia;
  constexpr bool kStatic = CellData<NMOL, NCIA>::kStatic;
  double e = 0.0;
  if (kStatic) {
#pragma unroll
    for (int m = 0; m < (kStatic ? NMOL : 0); m++) {
      const D2 wt = ld2(row + L::W + 2 * m);
      e = m == 0 ? wt.x * x.lo[0] : fma(wt.x, x.lo[m < CellData<NMOL, NCIA>::NG ? m : 0], e);
      e = fma(wt.y, x.hi[m < CellData<NMOL, NCIA>::NG ? m : 0], e);
    }
  } else {
    const size_t plane = (size_t)c.nwave * c.gms * 8;
    const char *lo = P.g + double_to_bits(row[L::GOFF]) + goff;
    const char *hi = lo + plane;
    for (int m = 0; m < ngmol; m++) {
      const D2 wt = ld2(row + L::W + 2 * m);
      e = m == 0 ? wt.x * ld1b(lo) : fma(wt.x, ld1b(lo + 8 * m), e);
      e = fma(wt.y, ld1b(hi + 8 * m), e);
    }
  }
  if (part == 1) return e;
  double ecs = 0.0;
  const double *cr = row + L::W + 2 * ngmol;
#pragma unroll
  for (int f = 0; f < (NCIA >= 0 ? NCIA : kMaxCia); f++) {
    if (f < ncia) {
      D4 q;
      if (CellData<NMOL, NCIA>::kStaticCia) q = x.q[f < CellData<NMOL, NCIA>::NC ? f : 0];
      else {
        const char *pq = P.cia[f] + double_to_bits(cr[6 * f]) + coff;
        const D2 k0 = ld2b(pq), k1 = ld2b(pq + 16);
        q.x = k0.x; q.y = k0.y; q.z = k1.x; q.w = k1.y;
      }
      const D2 cy = ld2(cr + 6 * f + 2), cz = ld2(cr + 6 * f + 4);
      double v = cy.x * q.x;
      v = fma(cy.y, q.z, v);
      v = fma(cz.x, q.y, v);
      v = fma(cz.y, q.w, v);
      if (hi_word(v) > 0) ecs += v;                            // v > 0 (crosssec.c:330)
    }
  }
  if (part == 2) return ecs;
  if (!SC) return e + ecs;                                     // = (e + 0 wn4) + 0 + ecs, to the bit
  const D2 sc = ld2(row + L::SCAT);                            // (scattering coefficient, cloud)
  return fma(sc.x, wn4, e) + sc.y + ecs;
}

template <int NMOL, int NCIA, bool SC = true>
BART_HD double cell_extinction(const DevConfig &c, const ColPtrs &P, const double *row, double wn4,
                               int part, size_t goff = 0, size_t coff = 0) {
  CellData<NMOL, NCIA> x;
  cell_load<NMOL, NCIA>(c, P, row, x, goff, coff);
  return cell_combine<NMOL, NCIA, SC>(c, P, row, x, wn4, part, goff, coff);
}

// ---------------------------------------------------------------------------------------
// Eclipse geometry, one (model, wavenumber) column: fused lookup + optical-depth scan +
// emergent intensity + hemispheric flux.
//   tau: eclipsetau eclipse.c:28-105 restated as a top-aligned Simpson prefix scan (the
//        reference re-integrates from each depth to the top; its panels are always aligned to
//        the top sample, numerical.c:454-525, so tau(d) = sum of completed panels (+ one
//        trapezoid when d is odd));  stop at the first tau > toomuch (tau.c:277-287).
//   intensity + flux: eclipse_intens eclipse.c:117-160 and flux eclipse.c:242-287 are
//        F = pi sum_a wgt_a [B_L d_L^a - 1/2 sum_i (d_{i+1}^a - d_i^a)(B_{i+1} + B_i)], d_i^a =
//        exp(-tau_i/mu_a).  The angle sum commutes with the layer sum, so the column carries
//        D_i = sum_a wgt_a d_i^a: F = pi [B_L D_L - 1/2 sum_i (D_{i+1} - D_i)(B_{i+1} + B_i)].
//        While every column of the warp has tau <= tau_small, D comes from its Maclaurin series
//        (one polynomial instead of one exp per angle).  The Planck prefactor 2 h c^2 wn^3 is
//        common to every layer of a column and is applied once, to the result.
// fp64 instruction budget per (depth, column) on the exponential branch (W12: 4 molecules, 1 CIA
// file, 5 angles with one squaring): extinction 15, tau 2.5, Planck 7 (one degree-4 exponential
// per thread, chained to the thread's other columns; reciprocal by seed + one Newton step), D 34
// (four degree-4 exponentials whose table factor carries the angle's weight, so the angle sum
// rides on their last multiply-add), layer sum 3, toomuch test 1.
// All 32 lanes of a warp must enter together (warp votes); a column that has passed its `last`
// layer idles until the warp's deepest column is done.  A thread carries NCOL independent
// columns of the same model, CSTRIDE samples apart starting at w0 (the table record of a depth is
// read once for all of them, and the independent dependency chains overlap); a column with
// valid[k] false idles from the start -- it may lie past the end of the spectrum: its loads are
// issued all the same (the launcher pads the grid and the CIA tables by NCOL CSTRIDE samples).
// etab: ecl_tab_entries(nang) entries (fill_ecl_exp_table).
// SQ >= 0 encodes (src << 4 | dst): the exponential of angle dst is the square of that of src
// (1/mu_dst = 2/mu_src, e.g. 60 and 0 degrees of the default ray grid); CHAIN: Planck chaining;
// With NCOL 1 and CHAIN, `upper` marks a column that the NCOL 2 form would carry as a thread's
// second one: its Planck exponential is then chained from the column CSTRIDE below in the same
// way, and -- the series-or-exponentials decision being taken per slot, i.e. per group of 32
// consecutive columns -- the result equals the NCOL 2 form's to the bit (small-batch kernel).
// PGEN: Planck exponent clamped per column and evaluated to degree 5 (DevConfig::planck_generic);
// SC false: no scattering and no cloud in any record of the launch (the terms are skipped).
// AHEAD: the grid and CIA samples of depth d + 1 are loaded during step d (the slot kernel: one warp
// per CTA, latency-bound); false: each step loads its own depth's samples (the throughput kernel,
// whose 20 warps per SM cover the latency; the samples are then not live across D(tau), the
// register peak of the step, which is what fits it in 96 registers).
template <int NMOL, int NCIA, int NANG, bool KEEP, int NCOL, int SQ = -1, bool CHAIN = false,
          int CSTRIDE = 0, bool PGEN = true, bool SC = true, bool AHEAD = true>
BART_HD void eclipse_columns(const DevConfig &c, const double *tab, const unsigned long long *etab,
                             int w0, const bool (&valid)[NCOL],
                             double *const (&tau_keep)[NCOL], int *const (&last_keep)[NCOL],
                             double (&flux)[NCOL], bool upper = false) {
  typedef TabLayout L;
  const int nl = c.nlayer;
  const int nf = c.lay.nf();
  const int nang = NANG > 0 ? NANG : c.nang;
  const int small_hi = hi_word(c.tau_small), clamp_hi = hi_word(c.tau_clamp);
  constexpr bool kStatic = CellData<NMOL, NCIA>::kStatic;
  const size_t gstep = (size_t)CSTRIDE * (kStatic ? CellData<NMOL, NCIA>::NG : c.gms) * 8;
  const size_t cstep = (size_t)CSTRIDE * 32;
  double wn4[NCOL], c2n[NCOL];
  double er1[NCOL], S[NCOL], trap[NCOL], Dprev[NCOL], Bprev[NCOL];
  int last[NCOL];
  bool alive[NCOL];
  const ColPtrs P = col_ptrs<NCIA>(c, w0);

  // Planck function without its prefactor, 1/(exp(hc wn/(k T)) - 1), of every column at one depth
  // (eclipse_intens, eclipse.c:130-140)
  auto planck = [&](const double *row, double (&B)[NCOL]) {
    double E = 0.0;
    const D2 tp = ld2(row + L::INVT);                          // (1/T, chaining factor)
#pragma unroll
    for (int k = 0; k < NCOL; k++) {
      double em1;
      if (CHAIN && k > 0) {
        em1 = fma(E, tp.y, -1.0);
        if (k + 1 < NCOL) E *= tp.y;
      } else {
        double it = tp.x;
        if (PGEN && it * c2n[k] > kExpYmax) it = kExpYmax / c2n[k];           // exponent <= 700
        if (CHAIN) {
          E = PGEN ? exp_core5(c2n[k], it, etab, 0.0) : exp_w(c2n[k], it, etab, 0.0);
          em1 = NCOL == 1 && upper ? fma(E, tp.y, -1.0) : E - 1.0;
        } else em1 = PGEN ? exp_core5(c2n[k], it, etab, -1.0) : exp_w(c2n[k], it, etab, -1.0);
      }
      B[k] = fast_rcp1(em1);
    }
  };

  // depth 0 (top): tau = 0, D = D(0)
#pragma unroll
  for (int k = 0; k < NCOL; k++) {
    const int wk = w0 + k * CSTRIDE;
    const double wn = c.wn[wk < c.nwave ? wk : c.nwave - 1];
    wn4[k] = (wn * wn) * (wn * wn);
    c2n[k] = cH * wn * cLS / cKB * kExpScale;                  // Planck exponent x N/ln2, per 1/T
    if (CHAIN && NCOL == 1 && upper) c2n[k] = cH * c.wn[wk - CSTRIDE] * cLS / cKB * kExpScale;
    S[k] = 0.0; trap[k] = 0.0; Dprev[k] = c.d0;
    alive[k] = valid[k] && !(0.0 > c.toomuch);
    last[k] = alive[k] ? nl - 1 : 0;
    if (KEEP && valid[k]) tau_keep[k][0] = 0.0;
  }
  planck(tab, Bprev);

  auto any_alive = [&]() {
    bool a = false;
#pragma unroll
    for (int k = 0; k < NCOL; k++) a = a || alive[k];
    return BART_WARP_ANY(a);
  };

  // The CIA samples of a column depend on the depth only through the bracket row of the layer's
  // temperature in the table's (coarse) temperature grid: consecutive layers mostly share it, so
  // cur[k].q is kept and reloaded only when a depth's row differs from `have` (warp-uniform test)
  CellData<NMOL, NCIA> cur[NCOL];
  CellOffs<NCIA> have = cell_offsets<NMOL, NCIA>(tab);                          // what cur[k].q holds
  auto fetch = [&](const CellOffs<NCIA> &o) {
    bool fresh = false;
#pragma unroll
    for (int f = 0; f < (NCIA > 0 ? NCIA : 0); f++) fresh = fresh || o.cia[f] != have.cia[f];
#pragma unroll
    for (int k = 0; k < NCOL; k++) cell_load_at<NMOL, NCIA>(c, P, o, cur[k], k * gstep, k * cstep, fresh);
    have = o;
  };
#pragma unroll
  for (int k = 0; k < NCOL; k++) cell_load<NMOL, NCIA>(c, P, tab, cur[k], k * gstep, k * cstep);
#pragma unroll
  for (int k = 0; k < NCOL; k++)
    er1[k] = cell_combine<NMOL, NCIA, SC>(c, P, tab, cur[k], wn4[k], false, k * gstep, k * cstep);
  // AHEAD: the loads of depth d + 1 are issued as soon as the data of depth d has been folded into
  // its extinction (same registers) and complete under the fp64 work of the rest of the step; their
  // addresses come from offsets read one step earlier still, so that no load instruction waits on
  // a shared-memory read.  Otherwise a step issues its own depth's loads first, ahead of the Planck
  // function, and folds them into the extinction before D(tau).
  const double *row_last = tab + (size_t)(nl - 1) * nf;
  auto row_after = [&](const double *r) { return r < row_last ? r + nf : r; };   // the bottom depth re-reads itself
  constexpr bool kLoadInStep = kStatic && !AHEAD;
  CellOffs<NCIA> offs;
  if (AHEAD) {
    fetch(cell_offsets<NMOL, NCIA>(row_after(tab)));
    offs = cell_offsets<NMOL, NCIA>(row_after(row_after(tab)));                 // of depth 2
  }

  auto step = [&](const double *row, int d, bool odd) {
    double tau[NCOL], B[NCOL], D[NCOL];
    bool small[NCOL];
    double erk[NCOL];
    if (kLoadInStep) {
      fetch(cell_offsets<NMOL, NCIA>(row));
      planck(row, B);
    }
#pragma unroll
    for (int k = 0; k < NCOL; k++) {
      erk[k] = cell_combine<NMOL, NCIA, SC>(c, P, row, cur[k], wn4[k], false, k * gstep, k * cstep);
    }
    if (AHEAD && kStatic) {
      fetch(offs);
      offs = cell_offsets<NMOL, NCIA>(row_after(row_after(row)));
    }
#pragma unroll
    for (int k = 0; k < NCOL; k++) {
      const double er = erk[k];
      if (odd) {
        tau[k] = fma(row[L::TR], er + er1[k], S[k]);
        // the panel that ends at depth d + 1 takes its terms of depths d - 1 and d now:
        // S(d+1) = SA er(d+1) + (SB er(d) + (SC er(d-1) + S(d-1))), so no er is carried
        // across the rest of this step
        const double *nx = row_after(row);
        S[k] = fma(nx[L::SB], er, fma(nx[L::SC], er1[k], S[k]));
      } else {
        S[k] = fma(row[L::SA], er, S[k]);
        tau[k] = S[k];
        er1[k] = er;
      }
      small[k] = !alive[k] || hi_word(tau[k]) < small_hi;
    }
    if (!kLoadInStep) planck(row, B);
    // D(tau): the low-tau polynomial while every live column of a slot (32 consecutive columns: the
    // warp's k-th) is below tau_small, weighted exponentials otherwise
    auto series = [&](int k0, int k1) {
#pragma unroll
      for (int k = 0; k < NCOL; k++)
        if (k >= k0 && k < k1) {
          const double u = fma(tau[k], c.ser_s, -1.0);
          double p = c.taylor[kTaylorN - 1];
#pragma unroll
          for (int i = kTaylorN - 2; i >= 0; i--) p = fma(p, u, c.taylor[i]);
          D[k] = p;
        }
    };
    auto exponentials = [&](int k0, int k1) {
      // exp arguments stay above -690: only the last depth of a column can exceed the clamp
      bool big = false;
      double tc[NCOL];
#pragma unroll
      for (int k = 0; k < NCOL; k++) { big = big || hi_word(tau[k]) >= clamp_hi; tc[k] = tau[k]; }
      if (BART_WARP_ANY(big)) {
#pragma unroll
        for (int k = 0; k < NCOL; k++) tc[k] = hi_word(tau[k]) >= clamp_hi ? c.tau_clamp : tau[k];
      }
      if (SQ >= 0) {
        // the source angle of the squaring first (its value is needed, not only its share of the
        // sum), then the others ride on the running sum
#pragma unroll
        for (int k = 0; k < NCOL; k++)
          if (k >= k0 && k < k1) {
            const double e = exp_w(tc[k], -c.exp_a[SQ >> 4], etab + (1 + (SQ >> 4)) * kExpTabSize, 0.0);
            D[k] = fma(e * e, c.sq_coef, e);
          }
      } else {
#pragma unroll
        for (int k = 0; k < NCOL; k++) if (k >= k0 && k < k1) D[k] = 0.0;
      }
#pragma unroll
      for (int a = 0; a < (NANG > 0 ? NANG : kMaxAng); a++)
        if (a < nang && !(SQ >= 0 && (a == (SQ >> 4) || a == (SQ & 15)))) {
#pragma unroll
          for (int k = 0; k < NCOL; k++)
            if (k >= k0 && k < k1) D[k] = exp_w(tc[k], -c.exp_a[a], etab + (1 + a) * kExpTabSize, D[k]);
        }
    };
    // one vote per slot (a single REDUX over a flag word measured slower: 4.48 vs 4.18 ms)
    unsigned sm = 0;                                           // bit k: slot k takes the series
#pragma unroll
    for (int k = 0; k < NCOL; k++) sm |= BART_WARP_ALL(small[k]) ? 1u << k : 0u;
    // (one decision for the whole warp instead of one per slot measured slower)
    if (sm == (1u << NCOL) - 1u) series(0, NCOL);
    else if (sm == 0u) exponentials(0, NCOL);
    else {                                                     // slots disagree (a few depths per column)
#pragma unroll
      for (int k = 0; k < NCOL; k++) { if (sm >> k & 1u) series(k, k + 1); else exponentials(k, k + 1); }
    }
#pragma unroll
    for (int k = 0; k < NCOL; k++)
      if (alive[k]) {
        if (KEEP) tau_keep[k][d] = tau[k];
        trap[k] = fma(D[k] - Dprev[k], B[k] + Bprev[k], trap[k]);
        Dprev[k] = D[k]; Bprev[k] = B[k];
        if (tau[k] > c.toomuch) { last[k] = d; alive[k] = false; }
      }
  };

  // the warp leaves the depth loop when all its columns have passed toomuch (checked every other
  // depth: a step on a finished column changes nothing)
  const double *row = tab + nf;
  for (int d = 1; d < nl; d += 2, row += 2 * nf) {
    if (!any_alive()) break;
    step(row, d, true);
    if (d + 1 >= nl) break;
    step(row + nf, d + 1, false);
  }
#pragma unroll
  for (int k = 0; k < NCOL; k++) {
    if (KEEP && valid[k]) *last_keep[k] = last[k];
    const int wk = w0 + k * CSTRIDE;
    const double wn = c.wn[wk < c.nwave ? wk : c.nwave - 1];
    const double c1 = 2.0 * cH * (wn * wn * wn) * cLS * cLS;
    flux[k] = cPI * c1 * (Bprev[k] * Dprev[k] - 0.5 * trap[k]);
  }
}

// single-column form (host emulation, tests)
template <int NMOL, int NCIA, int NANG, bool KEEP>
BART_HD double eclipse_column(const DevConfig &c, const double *tab, const unsigned long long *etab,
                              int w, double *tau_keep, int *last_keep) {
  const bool valid[1] = {true};
  double *const tk[1] = {tau_keep};
  int *const lk[1] = {last_keep};
  double flux[1];
  eclipse_columns<NMOL, NCIA, NANG, KEEP, 1>(c, tab, etab, w, valid, tk, lk, flux);
  return flux[0];
}

// ---------------------------------------------------------------------------------------
// Transit geometry.  Chord weights of one model, row d: tau(d) = sum_i wt[i] * er[i], i = 0..d,
// restating totaltau1 (slantpath.c:18-108): abscissa s_i = sqrt(r_i^2 - b^2) along the chord at
// impact parameter b = r(depth d), top-aligned Simpson panels with a trapezoid on the bottom
// interval when the count is even, the two-point case through the reference's 3-point
// construction, result x2 (both halves of the chord) and x rfct (tau.c:274).
// `W(i)` returns a reference to where the weight of depth i lives (packed row, or the tiled layout
// below).
// Every element of the row is stored exactly once (an element shared by two Simpson panels is the
// sum of the lower panel's bottom term, kept in a register, and the upper panel's top term, in
// that order -- the order the reference's accumulation gives), and a row can be split over
// `nparts` workers: part k takes a contiguous share of the row's panels, recomputing the one panel
// below its first for that carried term, and the last part the trailing element(s).  rad(i): radius
// of depth i.
template <class Acc, class Rad>
BART_HD void transit_weight_row_parts(const DevConfig &c, Rad rad, int d, Acc W, int part, int nparts) {
  if (d == 0) { if (part == 0) W(0) = 0.0; return; }
  const double b = rad(d);
  const double f = 2.0 * c.rfct;
  if (d == 1) {
    if (part != 0) return;
    const double rm = (rad(1) + rad(0)) / 2.0;
    const double s1 = sqrt(rm * rm - b * b), s2 = sqrt(rad(0) * rad(0) - b * b);
    const double h0 = s1, h1 = s2 - s1;
    const double hsum = h0 + h1, hratio = h1 / h0, hfactor = hsum * hsum / (h0 * h1);
    const double a0 = (2.0 - hratio) * hsum / 6.0, a1 = hfactor * hsum / 6.0,
                 a2 = (2.0 - 1.0 / hratio) * hsum / 6.0;
    W(1) = f * (a0 + 0.5 * a1);                              // bottom sample (depth 1)
    W(0) = f * (a2 + 0.5 * a1);
    return;
  }
  // s at depth i
  auto sdep = [&](int i) { return i == d ? 0.0 : sqrt(rad(i) * rad(i) - b * b); };
  // the three terms of the panel spanning depths 2p (top), 2p+1, 2p+2 (bottom)
  auto panel = [&](double sT, double sM, double sB, double &top, double &mid, double &bot) {
    const double h0 = sM - sB, h1 = sT - sM;
    const double hsum = h0 + h1, hratio = h1 / h0, hfactor = hsum * hsum / (h0 * h1);
    bot = f * (2.0 - hratio) * hsum / 6.0;
    mid = f * hfactor * hsum / 6.0;
    top = f * (2.0 - 1.0 / hratio) * hsum / 6.0;
  };
  const int P = d / 2;                                       // panels p = 0 .. P-1
  const int p0 = (int)((long long)P * part / nparts), p1 = (int)((long long)P * (part + 1) / nparts);
  const bool tail = part == nparts - 1;
  if (p0 == p1 && !tail) return;
  double sT = sdep(2 * p0), carry = 0.0;                     // carry: the term element 2 p0 has from panel p0 - 1
  if (p0 > 0) {
    double t, m, bt;
    panel(sdep(2 * p0 - 2), sdep(2 * p0 - 1), sT, t, m, bt);
    carry = 0.0 + bt;
  }
  for (int p = p0; p < p1; p++) {
    const double sM = sdep(2 * p + 1), sB = sdep(2 * p + 2);
    double top, mid, bot;
    panel(sT, sM, sB, top, mid, bot);
    W(2 * p) = carry + top;
    W(2 * p + 1) = 0.0 + mid;
    carry = 0.0 + bot;
    sT = sB;
  }
  if (!tail) return;
  if (d & 1) {                                               // even count: bottom trapezoid
    const double h = sdep(d - 1);
    W(d - 1) = carry + f * h / 2.0;
    W(d) = 0.0 + f * h / 2.0;
  } else W(d) = carry;
}
template <class Acc>
BART_HD void transit_weight_row_acc(const DevConfig &c, const double *tab, int d, Acc W, int part = 0,
                                    int nparts = 1) {
  const int nf = c.lay.nf();
  transit_weight_row_parts(c, [tab, nf](int i) { return tab[(size_t)i * nf + TabLayout::RAD]; }, d, W, part, nparts);
}

// packed row: wt[i], i = 0..d
BART_HD void transit_weight_row(const DevConfig &c, const double *tab, int d, double *wt) {
  transit_weight_row_acc(c, tab, d, [wt](int i) -> double & { return wt[i]; });
}

// Tiled layout of one model's chord weights for the tile kernel: depth chunks of kTrChunk; chunk
// ch holds rows i = 0 .. min(kTrChunk (ch+1), nl) - 1 (the layers a chord of that chunk can cross),
// each row kTrRow doubles = kTrChunk / kTrTD groups of (kTrTD weights + padding to 16 bytes):
// element (depth d, layer i) sits at chunk d / kTrChunk, row i, group (d % kTrChunk) / kTrTD,
// slot d % kTrTD; weights with i > d are zero.  One chunk is one contiguous block (one bulk copy)
// and a warp's kTrTD weights for layer i are one aligned 48-byte broadcast read.
constexpr int kTrChunk = 20, kTrTD = 5, kTrGroup = 6, kTrRow = (kTrChunk / kTrTD) * kTrGroup;
BART_HD int tr_rows(int nl, int ch) { const int r = kTrChunk * (ch + 1); return r < nl ? r : nl; }
BART_HD size_t tr_chunk_off(int nl, int ch) {
  size_t rows = 0;
  for (int k = 0; k < ch; k++) rows += tr_rows(nl, k);
  return rows * kTrRow;
}
BART_HD int tr_nchunks(int nl) { return (nl + kTrChunk - 1) / kTrChunk; }
BART_HD size_t tr_stride(int nl) { return tr_chunk_off(nl, tr_nchunks(nl)); }
// rad: radii by depth (the kernel's shared-memory copy); part / nparts: transit_weight_row_parts
BART_HD void transit_weight_row_tiled(const DevConfig &c, const double *rad, int d, double *wm,
                                      int part = 0, int nparts = 1) {
  const int ch = d / kTrChunk, dl = d % kTrChunk;
  double *base = wm + tr_chunk_off(c.nlayer, ch) + (dl / kTrTD) * kTrGroup + dl % kTrTD;
  transit_weight_row_parts(c, [rad](int i) { return rad[i]; }, d,
                           [base](int i) -> double & { return base[(size_t)i * kTrRow]; }, part, nparts);
}

// Layout of one model's chord weights for the tensor-core tile kernel (transit_mma_kernel): depth
// chunks of 16 rows; chunk ch is a dense row-major 16 x mm_rs(ch) block holding W[d][i] for the
// chunk's depths d and layers i = 0 .. 16 (ch + 1) - 1 (zero above the diagonal and in the rows past
// the last layer).  The row stride is 4 modulo 16 doubles, which makes the A-fragment read of
// mma.m8n8k4 (lane -> row lane/4, column lane%4) touch every bank pair exactly twice.
constexpr int kMmChunk = 16;
BART_HD int mm_nchunks(int nl) { return (nl + kMmChunk - 1) / kMmChunk; }
BART_HD int mm_rs(int ch) { return kMmChunk * (ch + 1) + 4; }
BART_HD size_t mm_chunk_off(int ch) { return (size_t)128 * ch * (ch + 1) + (size_t)64 * ch; }
BART_HD size_t mm_stride(int nl) { return mm_chunk_off(mm_nchunks(nl)); }
BART_HD void transit_weight_row_mm(const DevConfig &c, const double *rad, int d, double *wm,
                                   int part = 0, int nparts = 1) {
  const int ch = d / kMmChunk;
  double *base = wm + mm_chunk_off(ch) + (size_t)(d % kMmChunk) * mm_rs(ch);
  transit_weight_row_parts(c, [rad](int i) { return rad[i]; }, d,
                           [base](int i) -> double & { return base[i]; }, part, nparts);
}

// modulationm1 (slantpath.c:446-473), modlevel -1: the planet as an opaque disc whose radius is
// where tau reaches toomuch, by linear interpolation (interp_line, pu/src/numerical.c:203-211)
// between the last two impact parameters.  tau0/tau1: optical depths at depths last-1 and last,
// b0/b1 their impact parameters (cm).  Returns -1 when toomuch was not reached (the reference
// exits, slantpath.c:308-316).
BART_HD double modulation_m1(double tau0, double tau1, double b0, double b1, double toomuch,
                             double inv_srad2, int *status) {
  if (tau1 < toomuch) { *status |= REJ_NOTOOMUCH; return -1.0; }
  const double dx = tau1 - tau0;
  const double m = (b1 - b0) / dx;
  const double muchrad = b0 + (toomuch - tau0) * m;
  return muchrad * muchrad * inv_srad2;
}

// Transit column: tau(d) by the chord weights, stop at toomuch, then the modulation integral
// (modulation1, slantpath.c:350-436) as a top-aligned Simpson scan over impact parameter.
// `er` is per-thread scratch with stride `es` (shared memory in the kernel).
template <int NMOL, int NCIA, bool KEEP>
BART_HD double transit_column(const DevConfig &c, const double *tab, const unsigned long long *etab,
                              const double *wts, int w, double *er, int es, double *tau_keep,
                              int *last_keep, int *status) {
  typedef TabLayout L;
  const int nl = c.nlayer;
  const int nf = c.lay.nf();
  const double wn = c.wn[w];
  const double wn4 = (wn * wn) * (wn * wn);
  double S = 0.0, f1 = 0.0, f2 = 0.0, tau = 0.0, tau_prev = 0.0;
  int last = nl - 1;
  int d;
  const ColPtrs P = col_ptrs<NCIA>(c, w);
  for (d = 0; d < nl; d++) {
    const double *row = tab + (size_t)d * nf;
    er[(size_t)d * es] = cell_extinction<NMOL, NCIA>(c, P, row, wn4, false);
    const double *wr = wts + (size_t)d * (d + 1) / 2;
    tau_prev = tau;
    tau = 0.0;
    for (int i = 0; i <= d; i++) tau += wr[i] * er[(size_t)i * es];
    if (KEEP) tau_keep[d] = tau;
    const double bd = row[L::RAD] * c.rfct;
    const double fd = fast_exp_neg(-tau, etab) * bd;
    if (d >= 2 && !(d & 1)) S += row[L::SA] * fd + row[L::SB] * f1 + row[L::SC] * f2;
    f2 = f1; f1 = fd;
    if (tau > c.toomuch) { last = d; break; }
  }
  if (KEEP) *last_keep = last;
  if (c.modlevel == -1) {
    const int i0 = last > 0 ? last - 1 : 0;
    return modulation_m1(tau_prev, tau, tab[(size_t)i0 * nf + L::RAD] * c.rfct,
                         tab[(size_t)(i0 + 1) * nf + L::RAD] * c.rfct, c.toomuch,
                         c.inv_srad2, status);
  }
  int n;                                                       // number of integration points
  if (last < nl - 1) {
    const int dd = last + 1;                                   // appended zero-integrand point
    const double *row = tab + (size_t)dd * nf;
    if (dd >= 2 && !(dd & 1)) S += row[L::SB] * f1 + row[L::SC] * f2;
    f2 = f1; f1 = 0.0;
    n = dd + 1;
  } else n = nl;
  if (n < 3) { *status |= REJ_FEWPTS; return -1.0; }
  if (!(n & 1)) S += tab[(size_t)(n - 1) * nf + L::TR] * (f1 + f2);
  const double btop = tab[L::RAD] * c.rfct;
  double res = btop * btop - 2.0 * S;
  if (c.transparent) {
    const double maxtau = tau > c.toomuch ? tau : c.toomuch;
    const double bl = tab[(size_t)(n - 1) * nf + L::RAD] * c.rfct;
    res -= fast_exp_neg(-maxtau, etab) * bl * bl;
  }
  return res * c.inv_srad2;
}

}  // namespace bart
