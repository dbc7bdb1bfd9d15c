// builder.cu -- stage (d): the line-by-line opacity-grid builder (`transit --justOpacity`).
//
// Reference: calcprofiles / calcopacity (transit/src/opacity.c:218-427), getprofile and
// computemolext(permol=1) (transit/src/extinction.c:8-57, 281-529), voigtn / voigtxy
// (pu/src/voigt.c:132-200, 369-554).  The reference loops layers x temperatures x lines on one
// core; here:
//
//   K5  voigt_table_kernel     one thread per output bin of every unique (Doppler, Lorentz)
//                              profile: fine samples by the 3-region Pierluissi approximation,
//                              bin-averaged in float32 with the reference's operation order.
//   line_index_kernel          per line: wavenumber, oversampled/coarse bin indices with
//                              non-contracted IEEE ops (bit-exact indices).
//   group_spec / fix / mark    co-add grouping of neighbouring lines (extinction.c:450-462) --
//                              temperature independent, done once: the reference's sequential
//                              leader chain as speculative per-block walks + one fix-up walk,
//                              then scans and a fill (load_lines_device); the line list itself
//                              streams file -> pinned staging -> HBM without a host copy.
//   K6a+b strength_kmax_kernel per plane (temperature): ONE pass over the lines evaluates the two
//                              exponentials that serve both the strongest line per molecule
//                              (extinction.c:400-427) and the co-added group strengths (439-464);
//                              strength_count / block_scan / strength_fill then compact the
//                              groups that pass the weak-line cut (467-470), in order.  These
//                              do not depend on the layer: once per T, not per cell.
//   K6c widths_kernel          per (layer, isotope): Lorentz/Doppler widths, table indices, the
//                              carried Doppler index of the reference's sequential loop.
//   K6d accumulate_kernel      per (layer, 128-bin wavenumber tile): GATHER over the candidate
//                              groups -- no atomics, deterministic; the Voigt pool is stored
//                              phase-major so that the samples a line adds to consecutive bins
//                              (stride `wnosamp` in the reference's array) are contiguous.
//
// The temperature axis is the sharding axis (bart_build_opacity_slice): planes are independent.
#include "builder.hpp"
#include "cuda_host.hpp"
#include "device.cuh"
#include "column_math.cuh"
#include <cuda_runtime.h>
#include <cmath>
#include <cstring>
#include <algorithm>
#include <vector>
#include <map>
#include <string>
#include <chrono>
#include <cub/device/device_scan.cuh>
#include <cub/iterator/transform_input_iterator.cuh>

namespace bart {

constexpr int kMaxIso = 64;
constexpr int kAccThreads = 128;

struct CellIso;

// Plane / cell work buffers of run_planes, shared by the grid build and the line-by-line forward
// mode; sized per call (ensure_grow).
struct PlaneWork {
  DevBuf<double> T, tq, facfull, fac2, kmax, S;                        // per plane
  DevBuf<int> blk;
  DevBuf<long long> total, base, cisobeg;
  DevBuf<int> c_idx;                                                   // compact pool
  DevBuf<int> cell_plane;                                              // per cell
  DevBuf<long long> cell_out;
  DevBuf<CellIso> cellinfo;
  DevBuf<int> iso_spec, iso_out;                                       // static tables
  DevBuf<double> iso_mass, spec_mass, spec_radius;
};

struct BuilderState {
  // sampling
  int nwave = 0, osamp = 0, nlayer = 0, nspec = 0, niso = 0, ngmol = 0, ntemp = 0;
  long long nowns = 0;
  double wn_lo = 0, dwn = 0, odwn = 0;
  std::vector<double> temps;
  // isotopes
  std::vector<int> iso_spec, iso_gmol, gmol_id;
  std::vector<double> ziso;                 // [niso][ntemp]
  // lines / groups
  long long nlines = 0, ngroups = 0, neval = 0;
  DevBuf<double> d_c_wavn, d_c_elow, d_c_gf;      // grouped lines
  DevBuf<long long> d_gstart;                     // [ngroups+1]
  DevBuf<int> d_giown, d_gidwn;
  DevBuf<short> d_giso;
  DevBuf<double> d_gwavn;
  std::vector<long long> iso_gbeg;          // [niso+1] group range per isotope
  std::vector<int> h_iown;                  // per-line trace (leader bin, or -2-bin when co-added)
  DevBuf<int> d_trace;                      // the same trace when the grouping ran on the device
  // Voigt table
  int nDop = 0, nLor = 0;
  std::vector<double> aDop, aLor;
  std::vector<long long> prof_off, prof_size;     // [nDop*nLor] offset (floats) and half-size
  DevBuf<float> d_prof;
  long long prof_total = 0;
  DevBuf<double> d_aDop, d_aLor;
  DevBuf<long long> d_prof_off, d_prof_size;
  PlaneWork work;
  DevBuf<double> dens, out;                      // grid build: [cell][nspec], [cell][ngmol][nwave]
  std::vector<std::vector<double>> zspline; // [niso] second derivatives of Z(T) (line-by-line mode)
  bool lines_loaded = false, profiles_ready = false, grid_ready = false;
  // per-phase wall/device milliseconds (bart_builder_phase_ms)
  std::map<std::string, double> phase_ms;
};

// Times a phase of the build on stream `s` with CUDA events (the builder synchronises between
// phases anyway, so this costs nothing on the data path).
struct PhaseTimer {
  BuilderState *b; const char *name; cudaStream_t s; cudaEvent_t e0, e1;
  PhaseTimer(BuilderState *b_, const char *n, cudaStream_t s_) : b(b_), name(n), s(s_) {
    cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, s);
  }
  ~PhaseTimer() {
    cudaEventRecord(e1, s); cudaEventSynchronize(e1);
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    b->phase_ms[name] += ms;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
  }
};

// ---------------------------------------------------------------------------------------
// Voigt function K(x, y) sqrt(ln2/pi) / alphaD (pu/src/voigt.c:132-200) as float.  Region I
// (x < 3, y < 1.8): w(z) = exp(-z^2) (1 + (2i/sqrt(pi)) int_0^z exp(t^2) dt), the integral as its
// Maclaurin series sum_k z^(2k+1) / (k! (2k+1)) carried as the running power p_k = -i z^(2k+1)
// (the reference evaluates it in 80-bit long double; fp64 here: <= 1e-10 relative before the
// float32 rounding).  Regions II / III: Pierluissi's sums over poles, Re sum_j c_j / (z^2 - s_j) in
// real arithmetic.  Operation order as in the reference's expressions (1-ulp parity of the table).
__constant__ double c_ferf[64];               // 1 / (k! (2k + 1))
__constant__ double c_pole2[3][2] = {{0.46131350, 0.19016350}, {0.09999216, 1.78449270},
                                     {0.002883894, 5.52534370}};      // {weight, shift}, region II
__constant__ double c_pole3[2][2] = {{0.51242424, 0.27525510}, {0.05176536, 2.72474500}};

__device__ float voigtxy_dev(double x, double y, double alphaD) {
  const double norm = 0.46971863934982566689 / alphaD;               // sqrt(ln 2 / pi) / alphaD
  const double two_over_sqrtpi = 1.12837916709551257389;
  const double zre = x * x - y * y, zim = 2 * x * y;                 // z^2, z = x + i y
  if (x < 3 && y < 1.8) {
    double sn, cs;
    sincos(zim, &sn, &cs);
    const int nterms = (x < 1 ? 15 : (int)(6.842 * x + 8.0)) + 1;
    double pre = y, pim = -x;                                        // -i z
    double sre = pre, sim = pim;
    for (int k = 1; k <= nterms; k++) {
      const double nim = pre * zim + pim * zre;                      // (pre + i pim) z^2
      const double nre = pre * zre - pim * zim;
      sim += nim * c_ferf[k];
      sre += nre * c_ferf[k];
      pim = nim; pre = nre;
    }
    return (float)(norm * exp(-zre) * (cs * (1 - sre * two_over_sqrtpi) - sn * sim * two_over_sqrtpi));
  }
  const double im2 = zim * zim, xim = zim * x;
  if (x < 5 && y < 5) {
    const double d0 = zre - c_pole2[0][1], d1 = zre - c_pole2[1][1], d2 = zre - c_pole2[2][1];
    return (float)(norm * (c_pole2[0][0] * ((xim - d0 * y) / (d0 * d0 + im2)) +
                           c_pole2[1][0] * ((xim - d1 * y) / (d1 * d1 + im2)) +
                           c_pole2[2][0] * ((xim - d2 * y) / (d2 * d2 + im2))));
  }
  const double d0 = zre - c_pole3[0][1], d1 = zre - c_pole3[1][1];
  return (float)(norm * (c_pole3[0][0] * ((xim - d0 * y) / (d0 * d0 + im2)) +
                         c_pole3[1][0] * ((xim - d1 * y) / (d1 * d1 + im2))));
}

struct ProfJob {          // one unique profile
  long long off;          // offset into the float pool
  int nwn;                // 2*halfsize+1
  int ipo;                // fine intervals per bin (1 => adjacent average / quick)
  int quick;
  int osamp, K;           // pool layout: sample i of the profile is stored at (i % osamp) * K + i / osamp
  double dint, dwn_half, alphaL, alphaD;
};

// voigtn (voigt.c:369-483) + meanintegSimp/Trap (489-554): thread per output bin.
__global__ void voigt_table_kernel(const ProfJob *jobs, float *pool) {
  const ProfJob jb = jobs[blockIdx.y];
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= jb.nwn) return;
  const double y = 0.83255461115769775635 * jb.alphaL / jb.alphaD;
  const long long base = (long long)k * jb.ipo;
  auto sample = [&](long long i) {
    const double xx = 0.83255461115769775635 * fabs(jb.dint * (double)i - jb.dwn_half) / jb.alphaD;
    return voigtxy_dev(xx, y, jb.alphaD);
  };
  float out;
  if (jb.quick) out = sample(base);
  else if (jb.ipo & 1) {                       // even point count: trapezoid (meanintegTrap)
    float acc = 0;
    for (int i = 1; i < jb.ipo; i++) acc += sample(base + i);
    const float ends = sample(base) + sample(base + jb.ipo);
    out = (float)((acc + ends / 2.0) / (double)jb.ipo);
  } else {                                     // odd point count: Simpson (meanintegSimp)
    float acc = 0;
    for (int i = 1; i < jb.ipo; i += 2) acc += sample(base + i);
    acc *= 2;
    for (int i = 2; i < jb.ipo; i += 2) acc += sample(base + i);
    acc *= 2;
    acc += sample(base) + sample(base + jb.ipo);
    out = (float)(acc / (jb.ipo * 3.0));
  }
  // phase-major ("transposed") storage: the samples one line adds to consecutive coarse bins
  // (stride osamp in the reference's array, extinction.c:499-507) are contiguous here
  pool[jb.off + (long long)(k % jb.osamp) * jb.K + k / jb.osamp] = out;
}

// ---------------------------------------------------------------------------------------
// Per-line indices (extinction.c:431-447, 476).  Non-contracted IEEE operations so that the
// integer truncations and the nearest-node test see the same doubles as a plain C build.
__global__ void line_index_kernel(const double *wl, long long n, double wn_lo, double own_last,
                                  double odwn, double dwn, double *wavn_out, int *iown_out,
                                  int *idwn_out, unsigned char *inrange) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double wavn = __ddiv_rn(1.0, __dmul_rn(wl[i], 1e-4));
  wavn_out[i] = wavn;
  const bool in = !(wavn < wn_lo || wavn > own_last);
  inrange[i] = in ? 1 : 0;
  int iown = 0, idwn = 0;
  if (in) {
    iown = (int)__ddiv_rn(__dadd_rn(wavn, -wn_lo), odwn);
    const double v0 = __dadd_rn(wn_lo, __dmul_rn((double)iown, odwn));
    const double v1 = __dadd_rn(wn_lo, __dmul_rn((double)(iown + 1), odwn));
    if (fabs(__dadd_rn(wavn, -v1)) < fabs(__dadd_rn(wavn, -v0))) iown++;
    idwn = (int)__ddiv_rn(__dadd_rn(wavn, -wn_lo), dwn);
  }
  iown_out[i] = iown;
  idwn_out[i] = idwn;
}

// ---------------------------------------------------------------------------------------
// Co-add grouping on the device (extinction.c:450-462).  The reference walks the lines once: an
// in-range line that no earlier leader absorbed leads a group and absorbs the FOLLOWING lines of its
// isotope while |wavn - owns[iown_leader]| < odwn; the next leader is the first in-range line after
// the run.  Who leads depends on who led before -- a chain through the whole list -- but the chain
// forgets its past quickly: where it goes from a line depends on that line only, so two walks that
// ever stand on the same line coincide from there on.
//   1. group_spec_kernel   one thread per block of kGrpBlock lines walks the chain SPECULATIVELY
//                          from the block's first in-range line, marks the leaders it visits and
//                          records where it leaves the block;
//   2. group_fix_kernel    one thread follows the TRUE chain from the first in-range line of the
//                          list, block by block, only until it steps on a speculative mark (from
//                          there the block's speculative marks and exit are the true ones): a
//                          step or two per block, whatever the line density;
//   3. group_mark_kernel   one thread per line: the true leaders (fix-up marks, and speculative
//                          marks at or after their block's merge point) mark their runs.
// This IS the reference's walk for any input (no ordering assumed); a list on which the walks never
// merge would make step 2 sequential, so it gives up after a bounded number of steps and the caller
// takes the host walk.
constexpr int kGrpBlock = 4096;
__global__ void group_check_kernel(const short *iso, const unsigned char *inr, long long n, int niso,
                                   int *flags) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int is = iso[i];
  int f = 0;
  if (is < 0 || is >= niso) f |= 1;
  if (i > 0 && is < iso[i - 1]) f |= 2;
  if (f) atomicOr(flags, f);
}

struct GroupArgs {
  const double *wavn; const short *iso; const unsigned char *inr; const int *iown;
  long long n; double wn_lo, odwn;
};
__device__ __forceinline__ long long grp_run_end(const GroupArgs &a, long long ln) {
  const short is = a.iso[ln];
  const double vnode = __dadd_rn(a.wn_lo, __dmul_rn((double)a.iown[ln], a.odwn));
  long long e = ln + 1;
  while (e < a.n && a.iso[e] == is && fabs(a.wavn[e] - vnode) < a.odwn) e++;
  return e;
}
__device__ __forceinline__ long long grp_next_leader(const GroupArgs &a, long long e) {
  while (e < a.n && !a.inr[e]) e++;                  // out-of-range lines never lead
  return e;
}

__global__ void group_spec_kernel(GroupArgs a, long long nblocks, unsigned char *spec, long long *exit_of) {
  const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (b >= nblocks) return;
  const long long lo = b * kGrpBlock, hi = min(a.n, lo + kGrpBlock);
  long long ln = grp_next_leader(a, lo);
  while (ln < hi) {
    spec[ln] = 1;
    ln = grp_next_leader(a, grp_run_end(a, ln));
  }
  exit_of[b] = ln;
}

__global__ void group_fix_kernel(GroupArgs a, long long nblocks, const unsigned char *spec,
                                 const long long *exit_of, unsigned char *fixl, long long *merge_at,
                                 int *gave_up) {
  long long entry = grp_next_leader(a, 0);
  long long steps = 0;
  const long long limit = 8 * nblocks + (1 << 20);
  for (long long b = 0; b < nblocks; b++) {
    const long long hi = min(a.n, (b + 1) * kGrpBlock);
    long long ln = entry, m = a.n;
    while (ln < hi) {
      if (spec[ln]) { m = ln; break; }
      fixl[ln] = 1;
      ln = grp_next_leader(a, grp_run_end(a, ln));
      if (++steps > limit) { *gave_up = 1; return; }
    }
    merge_at[b] = m;
    entry = m < hi ? exit_of[b] : ln;
  }
}

// flag bit 0: leads a group; bit 1: member of a group (leader or absorbed)
__global__ void group_mark_kernel(GroupArgs a, const unsigned char *spec, const unsigned char *fixl,
                                  const long long *merge_at, unsigned char *flag, int *trace) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  if (!(fixl[i] || (spec[i] && i >= merge_at[i / kGrpBlock]))) return;
  const int io = a.iown[i];
  flag[i] = 3; trace[i] = io;
  const long long e = grp_run_end(a, i);
  for (long long k = i + 1; k < e; k++) { flag[k] = 2; trace[k] = -2 - io; }
}

// first group of every isotope = leaders before the first line whose isotope index is >= k
__global__ void group_isobeg_kernel(const short *iso, long long n, int niso, const long long *lrank,
                                    long long ngroups, long long *out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k > niso) return;
  long long lo = 0, hi = n;
  while (lo < hi) { const long long mid = (lo + hi) >> 1; if (iso[mid] < k) lo = mid + 1; else hi = mid; }
  out[k] = lo < n ? lrank[lo] : ngroups;
}

struct FlagBit {
  int bit;
  __host__ __device__ long long operator()(unsigned char f) const { return (f >> bit) & 1; }
};

__global__ void group_fill_kernel(const double *wavn, const double *elow, const double *gf,
                                  const short *iso, const int *iown, const int *idwn,
                                  const unsigned char *flag, const long long *lrank,
                                  const long long *mrank, long long n, long long *gstart, int *giown,
                                  int *gidwn, short *giso, double *gwavn, double *c_wavn,
                                  double *c_elow, double *c_gf) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned char f = flag[i];
  if (f & 2) {
    const long long c = mrank[i];
    c_wavn[c] = wavn[i]; c_elow[c] = elow[i]; c_gf[c] = gf[i];
    if (f & 1) {
      const long long g = lrank[i];
      gstart[g] = c; giown[g] = iown[i]; gidwn[g] = idwn[i]; giso[g] = iso[i]; gwavn[g] = wavn[i];
    }
  }
}

// A PLANE is one temperature: per-isotope factors, the strongest line per output molecule, and
// the ordered list of co-added groups that pass the weak-line cut at that temperature (the cut
// depends on T only, so it is taken once per plane and every layer of the plane walks the short
// list).  A CELL is one (plane, layer): densities -> widths -> one extinction row per output
// molecule.  The grid build has one plane per grid temperature with nlayer cells each; the
// line-by-line forward mode (tau.c:163-175,253-264 -> computemolext(permol=0)) has one plane per
// (model, layer) with a single cell.

constexpr int kCompactThreads = 256;

struct PlaneArgs {
  const long long *gstart; const short *giso; const double *wavn, *elow, *gf;
  long long ngroups;
  const double *plane_T, *plane_fac2 /*[P][niso]*/, *plane_facfull /*[P][niso]*/;
  const double *plane_tq;           // [P] -EXPCTE / T, divided once per plane on the host
  double *kmax /*[P][kMaxGridMol]*/;
  double *S /*[P][ngroups]*/;
  const int *iso_out;
  int niso, nout;
  double ethresh, wn_lo, own_last;
  int nblk;
};

// K6a+b pass 1, grid = (blocks of 256 groups, planes): ONE evaluation of the two exponentials of
// every line serves both reference passes -- the strongest individual in-range line per output
// molecule (extinction.c:400-427, expression order kept) and the co-added group strength
// (extinction.c:439-464: lines of a group summed in file order, then the isotope factor).
// table of the fp64 exp of column_math.cuh (fast_exp_neg: <= 1e-15 relative, 11 instructions
// instead of libdevice's ~30; the pass is 2 exponentials per line and nothing else)
__device__ unsigned long long b_exp_table[kExpTabSize];

constexpr int kPlanesPerThread = 4;   // planes that share one read of a line's (wavn, elow, gf)

__global__ void __launch_bounds__(kCompactThreads)
strength_kmax_kernel(PlaneArgs a, int nplanes) {
  __shared__ double s_max[kPlanesPerThread][kMaxGridMol];
  __shared__ unsigned long long s_etab[kExpTabSize];
  if (threadIdx.x < kExpTabSize) s_etab[threadIdx.x] = b_exp_table[threadIdx.x];
  const int p0 = blockIdx.y * kPlanesPerThread;
  const long long g = blockIdx.x * (long long)kCompactThreads + threadIdx.x;
  if (threadIdx.x < kPlanesPerThread * kMaxGridMol) (&s_max[0][0])[threadIdx.x] = 0.0;
  __syncthreads();
  if (g < a.ngroups) {
    const int iso = a.giso[g];
    double Tq[kPlanesPerThread], ff[kPlanesPerThread], pk[kPlanesPerThread], lmax[kPlanesPerThread];
#pragma unroll
    for (int q = 0; q < kPlanesPerThread; q++) {
      const int p = min(p0 + q, nplanes - 1);              // planes past the end shadow the last one
      Tq[q] = a.plane_tq[p];                               // -EXPCTE / T: no division in the kernel
      ff[q] = a.plane_facfull[(size_t)p * a.niso + iso];
      pk[q] = 0.0; lmax[q] = 0.0;
    }
    const long long b = a.gstart[g], e = a.gstart[g + 1];
    for (long long i = b; i < e; i++) {
      const double w = a.wavn[i], gf = a.gf[i], el = a.elow[i];
      const bool inr = !(w < a.wn_lo || w > a.own_last);
#pragma unroll
      for (int q = 0; q < kPlanesPerThread; q++) {
        const double e1 = fast_exp_neg(Tq[q] * el, s_etab);
        const double e2 = 1 - fast_exp_neg(Tq[q] * w, s_etab);
        const double term = gf * e1 * e2;
        pk[q] = (i == b) ? term : pk[q] + term;
        if (inr) lmax[q] = fmax(lmax[q], ff[q] * gf * e1 * e2);
      }
    }
    const int m = a.iso_out[iso];
#pragma unroll
    for (int q = 0; q < kPlanesPerThread; q++)
      if (p0 + q < nplanes) {
        const int p = p0 + q;
        a.S[(size_t)p * a.ngroups + g] = pk[q] * a.plane_fac2[(size_t)p * a.niso + iso];
        // the maximum only grows: a stale read can only cause a redundant atomic
        if (lmax[q] > *(volatile double *)&s_max[q][m])
          atomicMax((unsigned long long *)&s_max[q][m], (unsigned long long)__double_as_longlong(lmax[q]));
      }
  }
  __syncthreads();
  if (threadIdx.x < kPlanesPerThread * kMaxGridMol) {
    const int q = threadIdx.x / kMaxGridMol, m = threadIdx.x % kMaxGridMol;
    if (p0 + q < nplanes && m < a.nout && s_max[q][m] > 0)
      atomicMax((unsigned long long *)&a.kmax[(size_t)(p0 + q) * kMaxGridMol + m],
                (unsigned long long)__double_as_longlong(s_max[q][m]));
  }
}

// K6b pass 2: survivors of the weak-line cut (extinction.c:467-470) per block of 256 groups.
__global__ void __launch_bounds__(kCompactThreads)
strength_count_kernel(PlaneArgs a, int *blkcnt /*[P][nblk]*/) {
  const int p = blockIdx.y;
  const long long g = blockIdx.x * (long long)kCompactThreads + threadIdx.x;
  bool alive = false;
  if (g < a.ngroups)
    alive = !(a.S[(size_t)p * a.ngroups + g] <
              a.ethresh * a.kmax[(size_t)p * kMaxGridMol + a.iso_out[a.giso[g]]]);
  const int cnt = __syncthreads_count(alive);
  if (threadIdx.x == 0) blkcnt[(size_t)p * a.nblk + blockIdx.x] = cnt;
}

// exclusive scan of a plane's block counts (in place) and the plane total; block per plane
__global__ void __launch_bounds__(1024)
block_scan_kernel(int *blkcnt, int nblk, long long *total) {
  __shared__ int s_warp[32];
  __shared__ int s_carry;
  int *v = blkcnt + (size_t)blockIdx.x * nblk;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int base = 0; base < nblk; base += 1024) {
    const int i = base + threadIdx.x;
    const int x = i < nblk ? v[i] : 0;
    int inc = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += y; }
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    if (wid == 0) {
      int w = s_warp[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += y; }
      s_warp[lane] = w;
    }
    __syncthreads();
    const int carry = s_carry;
    const int excl = carry + (wid > 0 ? s_warp[wid - 1] : 0) + inc - x;
    if (i < nblk) v[i] = excl;
    __syncthreads();
    if (threadIdx.x == 1023) s_carry = carry + s_warp[31];
    __syncthreads();
  }
  if (threadIdx.x == 0) total[blockIdx.x] = s_carry;
}

// K6b pass 3: ordered compaction of the surviving groups of every plane into the pool (group
// numbers; bins, wavenumbers and strengths are read through them), and the per-isotope ranges of
// the compact list.
__global__ void __launch_bounds__(kCompactThreads)
strength_fill_kernel(PlaneArgs a, const int *blkoff /*[P][nblk]*/, const long long *plane_base,
                     int *c_idx, long long *cisobeg /*[P][niso+1]*/) {
  __shared__ int s_warp[kCompactThreads / 32];
  const int p = blockIdx.y;
  const long long g = blockIdx.x * (long long)kCompactThreads + threadIdx.x;
  bool alive = false;
  double S = 0.0;
  int iso = 0;
  if (g < a.ngroups) {
    iso = a.giso[g];
    S = a.S[(size_t)p * a.ngroups + g];
    alive = !(S < a.ethresh * a.kmax[(size_t)p * kMaxGridMol + a.iso_out[iso]]);
  }
  const unsigned bal = __ballot_sync(0xffffffffu, alive);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) s_warp[wid] = __popc(bal);
  __syncthreads();
  int pos = blkoff[(size_t)p * a.nblk + blockIdx.x] + __popc(bal & ((1u << lane) - 1u));
  for (int w = 0; w < wid; w++) pos += s_warp[w];
  if (g >= a.ngroups) return;
  if (alive) {
    const long long q = plane_base[p] + pos;
    c_idx[q] = (int)g;       // the list holds group numbers only: 4 bytes per survivor and plane
  }
  long long *cb = cisobeg + (size_t)p * (a.niso + 1);
  const int prev = g > 0 ? a.giso[g - 1] : -1;
  for (int i = prev + 1; i <= iso; i++) cb[i] = pos;
  if (g == a.ngroups - 1)
    for (int i = iso + 1; i <= a.niso; i++) cb[i] = pos + (alive ? 1 : 0);
}

struct CellIso {          // per (cell, isotope)
  double alphal, alphad;  // Lorentz width; Doppler width / wavenumber
  int ilor, idop0;        // table indices (idop0: at wn[0])
  int idop_carry;         // Doppler index used by lines below the re-pick threshold
  int hwbins;             // max profile half-width in coarse bins (+2) any group of the cell can have
  long long gsplit;       // first compact entry (absolute) with alphad*wavn/alphal < 0.1
};

__device__ int nearest_dev(const double *a, double v, int lo, int hi) {
  while (hi - lo > 1) {
    const int mid = (hi + lo) >> 1;
    if (a[mid] > v) hi = mid; else lo = mid;
  }
  if (hi == lo) return lo;
  return fabs(a[hi] - v) < fabs(a[lo] - v) ? hi : lo;
}

struct CellArgs {
  const int *cell_plane;            // [ncell]
  const double *cell_dens;          // [ncell][nspec] mass densities
  const long long *cell_out;        // [ncell] offset (doubles) of the cell's [nout][nwave] block
  const double *plane_T;
  const long long *plane_base, *cisobeg;
  const int *c_idx;                 // compact lists of surviving group numbers (all planes)
  const int *giown, *gidwn; const double *gwavn;   // per group: line-centre bins, wavenumber
  const double *S;                  // [plane][ngroups] strengths
  long long ngroups;
  int niso, nspec, nout, nwave, osamp, nDop, nLor;
  const int *iso_spec, *iso_out;
  const double *aDop, *aLor;
  const long long *prof_off, *prof_size;
  const float *pool;
  double wn0, own_last, dwn;
  int total_mode;                   // permol = 0: strengths times the isotope's species density
};

// K6c: widths and table indices per (cell, isotope) (extinction.c:365-396, 478-483).
__global__ void widths_kernel(CellArgs a, CellIso *cells, const double *spec_mass,
                              const double *spec_radius, const double *iso_mass) {
  const int ci = blockIdx.x, i = threadIdx.x;
  if (i >= a.niso) return;
  const int p = a.cell_plane[ci];
  const double T = a.plane_T[p];
  const double *density = a.cell_dens + (size_t)ci * a.nspec;
  const double fdoppler = sqrt(2 * kKB * T / kAMU) * kSQRTLN2 / kLS;
  const double florentz = sqrt(2 * kKB * T / kPI / kAMU) / (kAMU * kLS);
  double al = 0.0;
  for (int j = 0; j < a.nspec; j++) {
    const double cs = spec_radius[j] + spec_radius[a.iso_spec[i]];
    al += density[j] / spec_mass[j] * cs * cs * sqrt(1 / iso_mass[i] + 1 / spec_mass[j]);
  }
  al *= florentz;
  const double ad = fdoppler / sqrt(iso_mass[i]);
  CellIso c;
  c.alphal = al; c.alphad = ad;
  // the reference searches with hi = nDop / nLor (one past the end, extinction.c:394-395);
  // clamped to the last valid entry here
  c.idop0 = nearest_dev(a.aDop, ad * a.wn0, 0, a.nDop - 1);
  c.ilor = nearest_dev(a.aLor, al, 0, a.nLor - 1);
  // lines are sorted by decreasing wavenumber inside an isotope, so "alphad*wavn/alphal >= 0.1"
  // holds for a prefix of the isotope's (compact) groups
  const long long base = a.plane_base[p];
  const long long *cb = a.cisobeg + (size_t)p * (a.niso + 1);
  const long long gb = base + cb[i], ge = base + cb[i + 1];
  long long lo = gb, hi = ge;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (ad * a.gwavn[a.c_idx[mid]] / al >= 1e-1) lo = mid + 1; else hi = mid;
  }
  c.gsplit = lo;
  // the sequential loop keeps the Doppler index of the last line that was re-picked AND evaluated
  // (weak lines `continue` before the re-pick, extinction.c:467-483): the last compact entry of
  // the prefix
  c.idop_carry = lo > gb ? nearest_dev(a.aDop, ad * a.gwavn[a.c_idx[lo - 1]], 0, a.nDop - 1) : c.idop0;
  // widest profile any group of the cell can pick: Doppler indices between those of the two
  // ends of the spectrum (nearest_dev is monotonic), or the carried one
  const int dhi = nearest_dev(a.aDop, ad * a.own_last, 0, a.nDop - 1);
  long long hw = a.prof_size[(size_t)c.idop_carry * a.nLor + c.ilor];
  for (int d = c.idop0; d <= dhi; d++) hw = max(hw, a.prof_size[(size_t)d * a.nLor + c.ilor]);
  c.hwbins = (int)(hw / a.osamp) + 2;
  cells[(size_t)ci * a.niso + i] = c;
}

// K6d: accumulate.  CTA = (128-bin tile, cell), 4 warps.  For every isotope the candidate groups
// (compact entries whose leader bin lies within the widest profile the tile can see) are dealt to
// the warps in batches of 32, one group per lane: Doppler index, profile pointer, bin range
// clipped to the tile (extinction.c:476-497).  A batch whose groups span few bins (the usual
// case above ~1 bar: Doppler cores of 1-3 bins, ~1e3 lines per bin) is reduced LANE-PER-GROUP:
// for each bin of the span every lane evaluates its own group's sample and a shuffle butterfly
// sums the 32 values.  A batch that spans many bins (pressure-broadened layers) is walked
// LANE-PER-BIN: the groups are staged in shared memory and each one is spread over the lanes,
// bin = first + lane + 32 k.  Every warp adds into its own shared-memory row of 128 partial sums
// (no atomics); the rows are combined in warp order when the output molecule changes.  The
// result is deterministic and independent of how planes are batched; the order in which the
// terms of a bin are added differs from the reference's line order (relative effect ~1e-16).
struct StagedGroup {
  const float *prof;      // prof[j] is the sample this group adds to coarse bin j
  double S;
  int minj, maxj;         // bin range clipped to the tile (empty: minj > maxj)
  int pad0, pad1;
};
constexpr int kAccWarps = 8;
constexpr int kAccCta = 32 * kAccWarps;
constexpr int kNarrowSpan = 12;

__device__ __forceinline__ float ldg_f32(const float *p) {
  float v;
  asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// TILE = coarse bins per CTA (128, or 512 at high resolution: a pressure-broadened group then spans
// dozens of tiles, and every tile it touches pays the group's staging -- Doppler index search, bin
// range, profile pointer -- once; wider tiles pay it for four times the bin updates).
// 4 CTAs (32 warps) per SM at 64 registers.  Measured at the high-resolution shape (1e7 lines onto 1e5
// wavenumbers, ms per 2 planes): 1 CTA/SM 716, 2: 390, 3: 307, 4: 266, 5: 258, 6: 257, 8: 295 -- the
// kernel lives on warps in flight (its inner loop waits on scattered 512-byte profile segments served
// by the L2), while below 48 registers the spills eat the gain at the W12 shape (9.0 -> 9.3 -> 10.3 ms).
// What bounds it there (ncu profiles/r02_builder_accumulate_hr_v8.txt: 133 ms per plane, 3.2e11 bin
// updates): the L1 data stage at 57 % (a warp's 128 bytes of one profile row start at an arbitrary
// float, so every load is two wavefronts) with the issue slots at 51 %; one update is LDG + F2F + DFMA
// plus a quarter of the per-group address arithmetic.  Measured and dropped in round 2 (ms per 2
// planes, against 266-272): (i) every group reading phase 0 of its profile -- the bound of ANY
// reordering that would make co-resident groups share profile rows in the L1 (sorting the candidate
// groups by sub-bin phase): 235, i.e. the L2 latency the stall samples point at is worth 14 % at most;
// (ii) float -> double as one integer multiply-add (bits * 2^29 + bias, exact for the positive normal
// floats the Voigt pool holds) instead of F2F on the XU pipe: 272 vs 267, the conversion is not the
// limiter; (iii) splitting a batch into tile-covering and partial groups by ballot masks: 290 (the
// mask loops lose the unrolled loads); (iv) 256- and 512-bin tiles: 284 and 356.
#ifndef BART_ACC_MINB
#define BART_ACC_MINB 4
#endif
template <int TILE>
__global__ void __launch_bounds__(kAccCta, BART_ACC_MINB)
accumulate_kernel(CellArgs a, const CellIso *cells, double *out, int fast) {
  constexpr int kBinsPerLane = TILE / 32;
  __shared__ double s_acc[kAccWarps][TILE];
  __shared__ StagedGroup s_g[kAccWarps][32];
  __shared__ double s_aDop[128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // Tile-fastest launch order.  (Measured alternative, round 2: cell-fastest, so that the layers of
  // one plane walk the same candidate groups together and the group list is read from HBM once
  // instead of once per layer -- 49 GB -> <1 GB of DRAM reads per plane at 1e7 lines -- ran 1.6x
  // SLOWER: the kernel is bound by instructions per bin update, not by DRAM, and co-resident CTAs of
  // very different profile widths balance worse.)
  const int ci = blockIdx.y;
  const int j0 = blockIdx.x * TILE;
  const int jt_hi = min(j0 + TILE - 1, a.nwave - 1);
  const bool full_tile = j0 + TILE - 1 < a.nwave;
  const int p = a.cell_plane[ci];
  const long long base0 = a.plane_base[p];
  const long long *cb = a.cisobeg + (size_t)p * (a.niso + 1);
  const double *Sp = a.S + (size_t)p * a.ngroups;
  double *o = out + a.cell_out[ci];
  for (int k = threadIdx.x; k < a.nDop && k < 128; k += blockDim.x) s_aDop[k] = a.aDop[k];
  for (int k = threadIdx.x; k < kAccWarps * TILE; k += blockDim.x) (&s_acc[0][0])[k] = 0.0;
  __syncthreads();
  double *acc = s_acc[warp];
  double r[kBinsPerLane];                  // lane-per-bin partial sums of bins j0 + lane + 32 k
#pragma unroll
  for (int k = 0; k < kBinsPerLane; k++) r[k] = 0.0;
  // isotopes of one molecule are contiguous (TLI database order); a molecule that re-appears
  // continues from what was stored
  auto flush = [&](int m) {
#pragma unroll
    for (int k = 0; k < kBinsPerLane; k++) { acc[lane + 32 * k] += r[k]; r[k] = 0.0; }
    __syncthreads();
    for (int t = threadIdx.x; t < TILE; t += kAccCta) {
      double v = 0.0;
#pragma unroll
      for (int w = 0; w < kAccWarps; w++) { v += s_acc[w][t]; s_acc[w][t] = 0.0; }
      const int j = j0 + t;
      if (j < a.nwave) o[(size_t)m * a.nwave + j] += v;
    }
    __syncthreads();
  };
  int cur_mol = -1;
  for (int iso = 0; iso < a.niso; iso++) {
    const int m = a.iso_out[iso];
    if (m != cur_mol) {
      if (cur_mol >= 0) flush(cur_mol);
      cur_mol = m;
    }
    const long long gb = base0 + cb[iso], ge = base0 + cb[iso + 1];
    if (gb == ge) continue;
    const CellIso c = cells[(size_t)ci * a.niso + iso];
    const double dens = a.total_mode ? a.cell_dens[(size_t)ci * a.nspec + a.iso_spec[iso]] : 1.0;
    // tile-local half-width: candidates of the cell-level window have wavenumbers inside it, so
    // their Doppler indices lie between those of the window's ends
    int hwb = c.hwbins;
    {
      double wlo = a.wn0 + (double)(j0 - c.hwbins - 1) * a.dwn;
      double whi = a.wn0 + (double)(j0 + TILE + c.hwbins + 1) * a.dwn;
      if (wlo < a.wn0) wlo = a.wn0;
      if (whi > a.own_last) whi = a.own_last;
      const int dl = nearest_dev(s_aDop, c.alphad * wlo, 0, a.nDop - 1);
      const int dh = nearest_dev(s_aDop, c.alphad * whi, 0, a.nDop - 1);
      long long hw = a.prof_size[(size_t)c.idop_carry * a.nLor + c.ilor];
      for (int d = dl; d <= dh; d++) hw = max(hw, a.prof_size[(size_t)d * a.nLor + c.ilor]);
      hwb = min(hwb, (int)(hw / a.osamp) + 2);
    }
    // candidate range: leader coarse bins in [j0 - hw, j0 + TILE - 1 + hw]; idwn is non-increasing
    const int hi_bin = j0 + TILE - 1 + hwb, lo_bin = j0 - hwb;
    long long x = gb, y = ge;
    while (x < y) { const long long mid = (x + y) >> 1; if (a.gidwn[a.c_idx[mid]] > hi_bin) x = mid + 1; else y = mid; }
    const long long first = x;
    y = ge;
    while (x < y) { const long long mid = (x + y) >> 1; if (a.gidwn[a.c_idx[mid]] >= lo_bin) x = mid + 1; else y = mid; }
    const long long last = x;                                   // exclusive
    for (long long base = first + 32 * warp; base < last; base += 32 * kAccWarps) {
      const long long g = base + lane;
      StagedGroup sg;
      sg.prof = a.pool; sg.S = 0.0; sg.minj = (1 << 30); sg.maxj = -(1 << 30); sg.pad0 = sg.pad1 = 0;
      if (g < last) {
        const int gi = a.c_idx[g];
        int idop = c.idop_carry;
        if (g < c.gsplit) idop = nearest_dev(s_aDop, c.alphad * a.gwavn[gi], 0, a.nDop - 1);
        const size_t pi = (size_t)idop * a.nLor + c.ilor;
        const int ps = (int)a.prof_size[pi];
        const int iown = a.giown[gi], idwn = a.gidwn[gi];
        const int subw = iown - idwn * a.osamp;
        const int offset = iown - ps;
        // bins whose profile index osamp*j - offset lies in [0, 2 ps] (extinction.c:486-509)
        int mn = idwn - (ps - subw) / a.osamp, mx = idwn + (ps + subw) / a.osamp;
        while (a.osamp * mn - offset < 0) mn++;
        while (a.osamp * mx - offset > 2 * ps) mx--;
        // phase-major profile storage: index = phase * K + k, osamp*j - offset = k*osamp + phase
        const int bj0 = a.osamp * mn - offset;
        const int K = (2 * ps) / a.osamp + 1;
        sg.prof = a.pool + a.prof_off[pi] + (long long)(bj0 % a.osamp) * K + (bj0 / a.osamp - mn);
        sg.minj = max(mn, j0);
        sg.maxj = min(mx, jt_hi);
        if (sg.minj > sg.maxj) { sg.minj = (1 << 30); sg.maxj = -(1 << 30); }
        const double Sg = Sp[gi];
        sg.S = a.total_mode ? Sg * dens : Sg;                   // extinction.c:472-473
      }
      const int lo = __reduce_min_sync(0xffffffffu, sg.minj);
      const int hi = __reduce_max_sync(0xffffffffu, sg.maxj);
      if (hi < lo) continue;
      if (hi - lo < kNarrowSpan) {
        for (int bb = lo; bb <= hi; bb++) {
          double v = 0.0;
          if (bb >= sg.minj && bb <= sg.maxj) v = sg.S * (double)sg.prof[bb];
#pragma unroll
          for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
          if (lane == 0) acc[bb - j0] += v;
        }
      } else {
        __syncwarp();
        s_g[warp][lane] = sg;
        __syncwarp();
        const int cnt = (int)min((long long)32, last - base);
        // every staged group covers the whole tile (the usual batch where profiles are wide): a
        // counted loop without range tests, loads at immediate offsets from one pointer per group
        const bool mine_full = g >= last || (sg.minj == j0 && sg.maxj == jt_hi);
        if (fast && full_tile && __all_sync(0xffffffffu, mine_full)) {
#pragma unroll 8
          for (int q = 0; q < cnt; q++) {
            const float *pp = s_g[warp][q].prof + (j0 + lane);
            const double Sq = s_g[warp][q].S;
#pragma unroll
            for (int k = 0; k < kBinsPerLane; k++) r[k] = fma(Sq, (double)__ldg(pp + 32 * k), r[k]);
          }
        } else {
#pragma unroll 4
          for (int q = 0; q < cnt; q++) {
            const StagedGroup t = s_g[warp][q];
#pragma unroll
            for (int k = 0; k < kBinsPerLane; k++) {
              const int bb = j0 + lane + 32 * k;
              if (bb >= t.minj && bb <= t.maxj) r[k] += t.S * (double)t.prof[bb];
            }
          }
        }
      }
    }
  }
  if (cur_mol >= 0) flush(cur_mol);
}

// ---------------------------------------------------------------------------------------
// host side

static void setup_static(BuilderState *b, const Options &o, const Atmosphere &a, const Molecules &mol,
                         Tli &t, const std::vector<double> &wn) {
  b->nwave = (int)wn.size();
  b->osamp = o.wnosamp;
  b->nlayer = a.nlayer();
  b->nspec = a.nspec();
  b->wn_lo = wn[0];
  b->dwn = o.wndelt;
  b->odwn = o.wndelt / o.wnosamp;                                  // owns.d / owns.o
  b->nowns = (long long)(b->nwave - 1) * o.wnosamp + 1;            // makesample1, makesample.c:93
  if (b->nowns > 0x7fffffffLL)                                     // the reference's `int iown` too
    fail("wavenumber oversampling: %d samples x wnosamp %d exceeds the 32-bit line-bin index "
         "(extinction.c:322); lower wnosamp", b->nwave, o.wnosamp);
  b->niso = t.niso();
  if (b->niso > kMaxIso) fail("at most %d isotopes are supported", kMaxIso);
  // setimol (readlineinfo.c:249-278) and the molID list of calcopacity (opacity.c:353-361)
  b->iso_spec.assign(b->niso, -1);
  b->iso_gmol.assign(b->niso, -1);
  b->gmol_id.clear();
  for (int i = 0; i < b->niso; i++) {
    const std::string &mn = t.db[t.iso_db[i]].molname;
    for (int j = 0; j < a.nspec(); j++) if (a.species[j] == mn) b->iso_spec[i] = j;
    if (b->iso_spec[i] < 0) fail("TLI molecule '%s' is not among the atmospheric species.", mn.c_str());
    const int id = mol.id[b->iso_spec[i]];
    int g = -1;
    for (size_t k = 0; k < b->gmol_id.size(); k++) if (b->gmol_id[k] == id) g = (int)k;
    if (g < 0) { b->gmol_id.push_back(id); g = (int)b->gmol_id.size() - 1; }
    b->iso_gmol[i] = g;
  }
  b->ngmol = (int)b->gmol_id.size();
  if (b->ngmol > kMaxGridMol) fail("at most %d line-list molecules are supported", kMaxGridMol);
}

// temperature grid of the opacity file and the partition functions on it (opacity.c:297-339)
static void setup_grid_temps(BuilderState *b, const Options &o, const Tli &t) {
  b->temps = make_sampling(o.tlow, o.thigh, o.tempdelt, 1);        // maketempsample
  b->ntemp = (int)b->temps.size();
  if (b->temps.front() < t.tmin)
    fail("The opacity file attempted to sample a temperature (%.1f K) below the lowest allowed TLI "
         "temperature (%.1f K).", b->temps.front(), t.tmin);
  if (b->temps.back() > t.tmax)
    fail("The opacity file attempted to sample a temperature (%.1f K) beyond the highest allowed "
         "TLI temperature (%.1f K).", b->temps.back(), t.tmax);
  b->ziso.assign((size_t)b->niso * b->ntemp, 0.0);
  for (int i = 0; i < b->niso; i++) {
    const std::vector<double> &T = t.db[t.iso_db[i]].T;
    std::vector<double> z(T.size());
    spline_second_derivs(T.data(), t.iso_Z[i].data(), (long)T.size(), z.data());
    for (int k = 0; k < b->ntemp; k++)
      b->ziso[(size_t)i * b->ntemp + k] = spline_eval(z.data(), (long)T.size(), T.data(),
                                                      t.iso_Z[i].data(), b->temps[k]);
  }
  b->grid_ready = true;
}

// calcprofiles (opacity.c:218-277) + getprofile (extinction.c:8-57)
static void build_profiles(BuilderState *b, const Options &o, cudaStream_t s) {
  if (b->profiles_ready) return;
  b->nDop = o.ndop; b->nLor = o.nlor;
  if (b->nDop > 128) fail("at most 128 Doppler-width samples are supported");
  auto logspace = [](double lo, double hi, int n) {             // iomisc.c:1064-1083
    std::vector<double> v(n);
    const double l0 = log10(lo), l1 = log10(hi), st = (l1 - l0) / (n - 1.0);
    for (int i = 0; i < n; i++) v[i] = pow(10, l0 + i * st);
    return v;
  };
  b->aDop = logspace(o.dmin, o.dmax, b->nDop);
  b->aLor = logspace(o.lmin, o.lmax, b->nLor);
  const int np = b->nDop * b->nLor;
  b->prof_off.assign(np, 0); b->prof_size.assign(np, 0);
  std::vector<ProfJob> jobs;
  long long total = 0;
  const double dwn = b->odwn;
  const float ta = o.nwidth;
  for (int i = 0; i < b->nDop; i++)
    for (int j = 0; j < b->nLor; j++) {
      const int p = i * b->nLor + j;
      if (b->aDop[i] * 10.0 < b->aLor[j] && i != 0) {             // reuse the previous Doppler row
        b->prof_off[p] = b->prof_off[p - b->nLor];
        b->prof_size[p] = b->prof_size[p - b->nLor];
        continue;
      }
      const float dop = (float)b->aDop[i], lor = (float)b->aLor[j];   // PREC_VOIGT arguments
      double big = dop; if (big < lor) big = lor;
      const double wvgt = big * ta;
      int nvgt = 2 * (long)(wvgt / dwn + 0.5) + 1;
      if (nvgt < 2) nvgt = 3;
      if (nvgt > 2 * b->nowns) nvgt = 2 * (int)b->nowns + 1;
      ProfJob jb;
      jb.off = total; jb.nwn = nvgt;
      jb.osamp = b->osamp; jb.K = (nvgt - 1) / b->osamp + 1;
      jb.alphaL = lor; jb.alphaD = dop;
      jb.dwn_half = dwn * (long)(nvgt / 2);
      jb.quick = nvgt > 99999 ? 1 : 0;                            // _voigt_maxelements
      // voigtn's choice of the fine sampling (voigt.c:393-431)
      const double ddwn = 2.0 * jb.dwn_half / (nvgt - 1);
      double dint = jb.alphaD / 49.0;
      if (ddwn < dint || jb.quick) { jb.dint = ddwn; jb.ipo = 1; }
      else {
        int nint = (int)(ddwn / dint) + 1;
        if (nint & 1) nint++;
        const long long ntot = (long long)nvgt * nint + 1;
        jb.dint = 2.0 * jb.dwn_half / (double)(ntot - 1);
        jb.ipo = nint;
      }
      b->prof_off[p] = total;
      b->prof_size[p] = nvgt / 2;
      total += (long long)jb.osamp * jb.K;
      jobs.push_back(jb);
    }
  b->prof_total = total;
  b->d_prof.ensure(std::max<long long>(1, total));
  CUDA_OK(cudaMemsetAsync(b->d_prof.p, 0, std::max<long long>(1, total) * sizeof(float), s));
  // series coefficients 1/(n!(2n+1)) (the table of voigt.c:47-108)
  double ferf[64];
  long double fac = 1.0L;
  ferf[0] = 1.0;
  for (int n = 1; n < 64; n++) { fac *= n; ferf[n] = (double)(1.0L / (fac * (2 * n + 1))); }
  CUDA_OK(cudaMemcpyToSymbol(c_ferf, ferf, sizeof(ferf)));
  unsigned long long etab[kExpTabSize];
  fill_exp_table(etab);
  CUDA_OK(cudaMemcpyToSymbol(b_exp_table, etab, sizeof(etab)));
  DevBuf<ProfJob> d_jobs;
  upload(d_jobs, jobs);
  int maxn = 0;
  for (auto &j : jobs) maxn = std::max(maxn, j.nwn);
  // grid.y is limited to 65535 jobs; 60x60 profiles fit
  const int chunk = 32768;
  PhaseTimer pt(b, "voigt_table", s);
  for (size_t j0 = 0; j0 < jobs.size(); j0 += chunk) {
    const int nj = (int)std::min<size_t>(chunk, jobs.size() - j0);
    dim3 grid((maxn + 127) / 128, nj);
    voigt_table_kernel<<<grid, 128, 0, s>>>(d_jobs.p + j0, b->d_prof.p);
  }
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaStreamSynchronize(s));
  upload(b->d_aDop, b->aDop);
  upload(b->d_aLor, b->aLor);
  upload(b->d_prof_off, b->prof_off);
  upload(b->d_prof_size, b->prof_size);
  b->profiles_ready = true;
}

// One column slice set of the TLI file -> device through the pinned staging.  No host copy of the
// line list is kept (2.6 GB at 1e8 lines).
static void upload_file_column(int fd, const TliLineMap &m, long long col_off, int esize, void *d_dst,
                               PinnedStage &st, cudaStream_t s) {
  char *dst = (char *)d_dst;
  for (size_t i = 0; i < m.count.size(); i++) {
    long long off = col_off + m.first[i] * esize, left = m.count[i] * esize;
    while (left > 0) {
      const size_t chunk = (size_t)std::min<long long>(left, (long long)st.size());
      if (!st.put(fd, off, chunk, dst, s)) fail("TLI file: read failed");
      dst += chunk; off += (long long)chunk; left -= (long long)chunk;
    }
  }
}

// Lines -> device -> indices -> co-add groups, all on the device.  Returns false (nothing kept) when
// the line list is not sorted within an isotope: the caller then takes the host walk.
static bool load_lines_device(BuilderState *b, const Options &o, const Tli &t, double lo, double hi_hint,
                              cudaStream_t s) {
  auto t0 = std::chrono::steady_clock::now();
  auto lap = [&](const char *name) {
    auto now = std::chrono::steady_clock::now();
    b->phase_ms[name] += std::chrono::duration<double, std::milli>(now - t0).count();
    t0 = now;
  };
  TliLineMap m;
  map_tli_lines(o.linedb, t, lo, hi_hint, m);
  const long long n = m.total;
  const long long na = std::max<long long>(1, n);
  DevBuf<double> d_wl(na), d_elow(na), d_gf(na);
  DevBuf<short> d_iso(na);
  {
    PinnedStage st;
    const Fd fd(o.linedb.c_str(), O_RDONLY);
    if (fd < 0) fail("Data file '%s' not found.", o.linedb.c_str());
    upload_file_column(fd, m, m.wl_off, 8, d_wl.p, st, s);
    upload_file_column(fd, m, m.iso_off, 2, d_iso.p, st, s);
    upload_file_column(fd, m, m.el_off, 8, d_elow.p, st, s);
    upload_file_column(fd, m, m.gf_off, 8, d_gf.p, st, s);
    CUDA_OK(cudaStreamSynchronize(s));
  }
  lap("read_tli_host");
  DevBuf<double> d_wavn(na);
  DevBuf<int> d_iown(na), d_idwn(na);
  DevBuf<unsigned char> d_inr(na);
  const long long nblocks = (na + kGrpBlock - 1) / kGrpBlock;
  DevBuf<unsigned char> d_spec(na), d_fixl(na), d_flag(na);
  DevBuf<int> d_trace(na), d_flags(1);
  DevBuf<long long> d_exit(nblocks), d_merge(nblocks), d_lrank(na + 1), d_mrank(na + 1);
  const double own_last = b->wn_lo + (double)(b->nowns - 1) * b->odwn;
  const unsigned grid = (unsigned)((na + 255) / 256);
  CUDA_OK(cudaMemsetAsync(d_flags.p, 0, 4, s));
  CUDA_OK(cudaMemsetAsync(d_spec.p, 0, na, s));
  CUDA_OK(cudaMemsetAsync(d_fixl.p, 0, na, s));
  CUDA_OK(cudaMemsetAsync(d_flag.p, 0, na, s));
  CUDA_OK(cudaMemsetAsync(d_trace.p, 0xff, na * 4, s));               // -1: in no group
  int flags = 0;
  if (n > 0) {
    line_index_kernel<<<grid, 256, 0, s>>>(d_wl.p, n, b->wn_lo, own_last, b->odwn, b->dwn, d_wavn.p, d_iown.p,
                                           d_idwn.p, d_inr.p);
    group_check_kernel<<<grid, 256, 0, s>>>(d_iso.p, d_inr.p, n, b->niso, d_flags.p);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaMemcpyAsync(&flags, d_flags.p, 4, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaStreamSynchronize(s));
  }
  if (flags & 1) fail("a TLI line has an isotope index outside [0,%d)", b->niso);
  if (flags & 2) fail("TLI lines are not grouped by isotope");
  long long ngroups = 0, nmember = 0;
  if (n > 0) {
    GroupArgs ga{d_wavn.p, d_iso.p, d_inr.p, d_iown.p, n, b->wn_lo, b->odwn};
    group_spec_kernel<<<(unsigned)((nblocks + 127) / 128), 128, 0, s>>>(ga, nblocks, d_spec.p, d_exit.p);
    group_fix_kernel<<<1, 1, 0, s>>>(ga, nblocks, d_spec.p, d_exit.p, d_fixl.p, d_merge.p, d_flags.p);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaMemcpyAsync(&flags, d_flags.p, 4, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaStreamSynchronize(s));
    if (flags) return false;                       // the walks never merged: host path
    group_mark_kernel<<<grid, 256, 0, s>>>(ga, d_spec.p, d_fixl.p, d_merge.p, d_flag.p, d_trace.p);
    CUDA_OK(cudaGetLastError());
    // ranks of the leaders (group numbers) and of the members (positions in the grouped line
    // arrays): exclusive sums over n + 1 flags, the last entry being the total
    cub::TransformInputIterator<long long, FlagBit, const unsigned char *> lead(d_flag.p, FlagBit{0}),
        memb(d_flag.p, FlagBit{1});
    size_t tmp_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, lead, d_lrank.p, n, s);
    DevBuf<char> d_tmp(std::max<size_t>(1, tmp_bytes));
    cub::DeviceScan::ExclusiveSum(d_tmp.p, tmp_bytes, lead, d_lrank.p, n, s);
    cub::DeviceScan::ExclusiveSum(d_tmp.p, tmp_bytes, memb, d_mrank.p, n, s);
    CUDA_OK(cudaGetLastError());
    long long lastr[2];
    unsigned char lastf = 0;
    CUDA_OK(cudaMemcpyAsync(&lastr[0], d_lrank.p + (n - 1), 8, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaMemcpyAsync(&lastr[1], d_mrank.p + (n - 1), 8, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaMemcpyAsync(&lastf, d_flag.p + (n - 1), 1, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaStreamSynchronize(s));
    ngroups = lastr[0] + (lastf & 1);
    nmember = lastr[1] + ((lastf >> 1) & 1);
  }
  b->nlines = n;
  b->ngroups = ngroups;
  b->d_gstart.ensure(ngroups + 1);
  b->d_giown.ensure(std::max<long long>(1, ngroups));
  b->d_gidwn.ensure(std::max<long long>(1, ngroups));
  b->d_giso.ensure(std::max<long long>(1, ngroups));
  b->d_gwavn.ensure(std::max<long long>(1, ngroups));
  b->d_c_wavn.ensure(std::max<long long>(1, nmember));
  b->d_c_elow.ensure(std::max<long long>(1, nmember));
  b->d_c_gf.ensure(std::max<long long>(1, nmember));
  if (n > 0) {
    group_fill_kernel<<<grid, 256, 0, s>>>(d_wavn.p, d_elow.p, d_gf.p, d_iso.p, d_iown.p, d_idwn.p, d_flag.p,
                                           d_lrank.p, d_mrank.p, n, b->d_gstart.p, b->d_giown.p, b->d_gidwn.p,
                                           b->d_giso.p, b->d_gwavn.p, b->d_c_wavn.p, b->d_c_elow.p, b->d_c_gf.p);
    CUDA_OK(cudaGetLastError());
  }
  CUDA_OK(cudaMemcpyAsync(b->d_gstart.p + ngroups, &nmember, 8, cudaMemcpyHostToDevice, s));
  b->iso_gbeg.assign(b->niso + 1, ngroups);
  if (n > 0) {
    DevBuf<long long> d_gbeg(b->niso + 1);
    group_isobeg_kernel<<<1, 128, 0, s>>>(d_iso.p, n, b->niso, d_lrank.p, ngroups, d_gbeg.p);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaMemcpyAsync(b->iso_gbeg.data(), d_gbeg.p, (b->niso + 1) * 8, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaStreamSynchronize(s));
  }
  CUDA_OK(cudaStreamSynchronize(s));
  b->h_iown.clear();
  b->d_trace = std::move(d_trace);
  lap("grouping_device");
  return true;
}

static void load_lines(BuilderState *b, const Options &o, Tli &t, const std::vector<double> &wn,
                       cudaStream_t s) {
  if (b->lines_loaded) return;
  double lo = wn.front(), hi_hint;
  // readdatarng selects with the HINTED limits wns.i / wns.f (readlineinfo.c:435-436)
  hi_hint = o.wnhigh > 0 ? o.wnhigh * o.wnfct : 1.0 / (o.wllow * o.wlfct);
  const char *force_host = getenv("BART_GROUP_HOST");
  if (!(force_host && atoi(force_host) != 0) && load_lines_device(b, o, t, lo, hi_hint, s)) {
    b->lines_loaded = true;
    return;
  }
  auto tp0 = std::chrono::steady_clock::now();
  read_tli_lines(o.linedb, t, lo, hi_hint);
  auto tp1 = std::chrono::steady_clock::now();
  b->phase_ms["read_tli_host"] += std::chrono::duration<double, std::milli>(tp1 - tp0).count();
  const long long n = (long long)t.wl.size();
  b->nlines = n;
  auto lap = [&](const char *name, std::chrono::steady_clock::time_point &from) {
    auto now = std::chrono::steady_clock::now();
    b->phase_ms[name] += std::chrono::duration<double, std::milli>(now - from).count();
    from = now;
  };
  auto tl = std::chrono::steady_clock::now();
  // the raw per-line arrays live until the grouped copies are on the device
  DevBuf<double> d_wl, d_elow, d_gf;
  DevBuf<short> d_isoid;
  upload(d_wl, t.wl); upload(d_elow, t.elow); upload(d_gf, t.gf);
  upload(d_isoid, t.isoid);
  const long long na = std::max<long long>(1, n);
  DevBuf<double> d_wavn(na);
  DevBuf<int> d_iown(na), d_idwn(na);
  DevBuf<unsigned char> d_inrange(na);
  const double own_last = b->wn_lo + (double)(b->nowns - 1) * b->odwn;
  if (n > 0) {
    line_index_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(d_wl.p, n, b->wn_lo, own_last, b->odwn,
                                                                   b->dwn, d_wavn.p, d_iown.p, d_idwn.p,
                                                                   d_inrange.p);
    CUDA_OK(cudaGetLastError());
  }
  std::vector<double> wavn(n);
  std::vector<int> iown(n), idwn(n);
  std::vector<unsigned char> inr(n);
  CUDA_OK(cudaStreamSynchronize(s));
  if (n > 0) {
    CUDA_OK(cudaMemcpy(wavn.data(), d_wavn.p, n * 8, cudaMemcpyDeviceToHost));
    CUDA_OK(cudaMemcpy(iown.data(), d_iown.p, n * 4, cudaMemcpyDeviceToHost));
    CUDA_OK(cudaMemcpy(idwn.data(), d_idwn.p, n * 4, cudaMemcpyDeviceToHost));
    CUDA_OK(cudaMemcpy(inr.data(), d_inrange.p, n, cudaMemcpyDeviceToHost));
  }
  lap("lines_h2d_index_d2h", tl);
  // co-add grouping (extinction.c:450-462): a leader absorbs the following lines of the same
  // isotope while |wavn - owns[iown_leader]| < odwn.  Out-of-range lines never lead, but are
  // absorbed when they follow a leader (the reference does not re-test the range in its while
  // loop).  The grouping does not depend on temperature or layer, so it is done once, here.
  auto tg0 = std::chrono::steady_clock::now();
  std::vector<long long> bounds;            // [ngroups+1] into the grouped line arrays
  std::vector<int> giown, gidwn;
  std::vector<short> giso;
  std::vector<double> gwavn, c_wavn, c_elow, c_gf;
  c_wavn.reserve(n); c_elow.reserve(n); c_gf.reserve(n);
  b->h_iown.assign(n, -1);
  b->iso_gbeg.assign(b->niso + 1, 0);
  int prev_iso = -1;
  for (long long ln = 0; ln < n; ln++) {
    const int iso = t.isoid[ln];
    if (iso < 0 || iso >= b->niso) fail("TLI line %lld has isotope index %d outside [0,%d)", ln, iso, b->niso);
    if (iso != prev_iso) {
      if (iso < prev_iso) fail("TLI lines are not grouped by isotope");
      for (int k = prev_iso + 1; k <= iso; k++) b->iso_gbeg[k] = (long long)giown.size();
      prev_iso = iso;
    }
    if (!inr[ln]) continue;
    const int io = iown[ln];
    const double vnode = b->wn_lo + (double)io * b->odwn;
    long long e = ln + 1;
    while (e < n && t.isoid[e] == iso && std::fabs(wavn[e] - vnode) < b->odwn) e++;
    bounds.push_back((long long)c_wavn.size());
    for (long long k = ln; k < e; k++) {
      c_wavn.push_back(wavn[k]); c_elow.push_back(t.elow[k]); c_gf.push_back(t.gf[k]);
    }
    giown.push_back(io); gidwn.push_back(idwn[ln]); giso.push_back((short)iso); gwavn.push_back(wavn[ln]);
    b->h_iown[ln] = io;
    for (long long k = ln + 1; k < e; k++) b->h_iown[k] = -2 - io;
    ln = e - 1;
  }
  bounds.push_back((long long)c_wavn.size());
  for (int k = prev_iso + 1; k <= b->niso; k++) b->iso_gbeg[k] = (long long)giown.size();
  b->ngroups = (long long)giown.size();
  b->phase_ms["grouping_host"] += std::chrono::duration<double, std::milli>(
      std::chrono::steady_clock::now() - tg0).count();
  tl = std::chrono::steady_clock::now();
  upload(b->d_gstart, bounds);
  upload(b->d_giown, giown); upload(b->d_gidwn, gidwn); upload(b->d_giso, giso);
  upload(b->d_gwavn, gwavn);
  upload(b->d_c_wavn, c_wavn); upload(b->d_c_elow, c_elow); upload(b->d_c_gf, c_gf);
  lap("groups_h2d", tl);
  b->lines_loaded = true;
}

// ---------------------------------------------------------------------------------------
// Plane / cell driver shared by the grid build and the line-by-line forward mode.

static void upload_statics(BuilderState *b, const Molecules &mol, const Tli &t, bool total_mode,
                           cudaStream_t s) {
  PlaneWork &w = b->work;
  std::vector<int> iso_out = b->iso_gmol;
  if (total_mode) std::fill(iso_out.begin(), iso_out.end(), 0);      // permol = 0: m stays 0
  CUDA_OK(cudaMemcpyAsync(w.iso_spec.ensure_grow(b->niso), b->iso_spec.data(), b->niso * 4, cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaMemcpyAsync(w.iso_out.ensure_grow(b->niso), iso_out.data(), b->niso * 4, cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaMemcpyAsync(w.iso_mass.ensure_grow(b->niso), t.iso_mass.data(), b->niso * 8, cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaMemcpyAsync(w.spec_mass.ensure_grow(b->nspec), mol.mass.data(), b->nspec * 8, cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaMemcpyAsync(w.spec_radius.ensure_grow(b->nspec), mol.radius_cm.data(), b->nspec * 8, cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaStreamSynchronize(s));
}

// Runs nplanes planes / ncell cells.  plane_T[P]; plane_Z[P][niso] partition functions;
// cell_plane[ncell] (non-decreasing); d_cell_dens[ncell][nspec] (device, mass densities);
// cell_out[ncell] offsets (doubles) into d_out of each cell's [nout][nwave] block, nout = ngmol
// (grid build) or 1 (total_mode).  Returns the number of evaluated (group, cell) pairs.
static long long run_planes(BuilderState *b, const Options &o, const Molecules &mol, const Tli &t,
                            int nplanes, const double *plane_T, const double *plane_Z, int ncell,
                            const int *cell_plane, const double *d_cell_dens,
                            const long long *cell_out, double *d_out, bool total_mode,
                            cudaStream_t s) {
  PlaneWork &w = b->work;
  upload_statics(b, mol, t, total_mode, s);
  const int niso = b->niso, nout = total_mode ? 1 : b->ngmol;
  const int nblk = (int)((b->ngroups + kCompactThreads - 1) / kCompactThreads);
  // per-isotope factors: pass 1 (extinction.c:412-418) uses ratio*SIGCTE*.../mass/Z per line,
  // pass 2 (464) SIGCTE*ratio/(mass*Z) per group
  std::vector<double> facfull((size_t)nplanes * niso), fac2((size_t)nplanes * niso);
  for (int p = 0; p < nplanes; p++)
    for (int i = 0; i < niso; i++) {
      const double Z = plane_Z[(size_t)p * niso + i];
      facfull[(size_t)p * niso + i] = t.iso_ratio[i] * kSIGCTE / t.iso_mass[i] / Z;
      fac2[(size_t)p * niso + i] = kSIGCTE * t.iso_ratio[i] / (t.iso_mass[i] * Z);
    }
  double *d_T = w.T.ensure_grow(nplanes), *d_facfull = w.facfull.ensure_grow(facfull.size()),
         *d_fac2 = w.fac2.ensure_grow(fac2.size()), *d_kmax = w.kmax.ensure_grow((size_t)nplanes * kMaxGridMol);
  int *d_blk = w.blk.ensure_grow((size_t)nplanes * std::max(1, nblk));
  long long *d_total = w.total.ensure_grow(nplanes), *d_base = w.base.ensure_grow(nplanes),
            *d_cisobeg = w.cisobeg.ensure_grow((size_t)nplanes * (niso + 1));
  CUDA_OK(cudaMemcpyAsync(d_T, plane_T, nplanes * 8, cudaMemcpyHostToDevice, s));
  std::vector<double> tq(nplanes);
  for (int p = 0; p < nplanes; p++) tq[p] = -kEXPCTE / plane_T[p];
  double *d_tq = w.tq.ensure_grow(nplanes);
  CUDA_OK(cudaMemcpyAsync(d_tq, tq.data(), nplanes * 8, cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaMemcpyAsync(d_facfull, facfull.data(), facfull.size() * 8, cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaMemcpyAsync(d_fac2, fac2.data(), fac2.size() * 8, cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaMemsetAsync(d_kmax, 0, (size_t)nplanes * kMaxGridMol * 8, s));
  CUDA_OK(cudaMemsetAsync(d_cisobeg, 0, (size_t)nplanes * (niso + 1) * 8, s));
  CUDA_OK(cudaMemsetAsync(d_total, 0, (size_t)nplanes * 8, s));
  const int *d_iso_out = w.iso_out.p;
  PlaneArgs pa;
  pa.gstart = b->d_gstart.p; pa.giso = b->d_giso.p; pa.wavn = b->d_c_wavn.p; pa.elow = b->d_c_elow.p;
  pa.gf = b->d_c_gf.p;
  pa.ngroups = b->ngroups; pa.plane_T = d_T; pa.plane_fac2 = d_fac2; pa.plane_facfull = d_facfull;
  pa.plane_tq = d_tq;
  pa.kmax = d_kmax; pa.S = w.S.ensure_grow((size_t)nplanes * std::max<long long>(1, b->ngroups));
  pa.iso_out = d_iso_out; pa.niso = niso; pa.nout = nout; pa.ethresh = o.ethreshold; pa.nblk = nblk;
  pa.wn_lo = b->wn_lo; pa.own_last = b->wn_lo + (double)(b->nowns - 1) * b->odwn;
  std::vector<long long> total(nplanes, 0), base(nplanes, 0);
  long long pool = 0;
  if (b->ngroups > 0) {
    PhaseTimer pt(b, "strength", s);
    strength_kmax_kernel<<<dim3(nblk, (nplanes + kPlanesPerThread - 1) / kPlanesPerThread), kCompactThreads, 0, s>>>(pa, nplanes);
    strength_count_kernel<<<dim3(nblk, nplanes), kCompactThreads, 0, s>>>(pa, d_blk);
    block_scan_kernel<<<nplanes, 1024, 0, s>>>(d_blk, nblk, d_total);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaMemcpyAsync(total.data(), d_total, nplanes * 8, cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaStreamSynchronize(s));
    for (int p = 0; p < nplanes; p++) { base[p] = pool; pool += total[p]; }
    CUDA_OK(cudaMemcpyAsync(d_base, base.data(), nplanes * 8, cudaMemcpyHostToDevice, s));
    int *ci = w.c_idx.ensure_grow(pool);
    strength_fill_kernel<<<dim3(nblk, nplanes), kCompactThreads, 0, s>>>(pa, d_blk, d_base, ci, d_cisobeg);
    CUDA_OK(cudaGetLastError());
  } else {
    CUDA_OK(cudaMemsetAsync(d_base, 0, nplanes * 8, s));
    w.c_idx.ensure_grow(1);
  }
  int *d_cell_plane = w.cell_plane.ensure_grow(ncell);
  long long *d_cell_out = w.cell_out.ensure_grow(ncell);
  CellIso *cells = w.cellinfo.ensure_grow((size_t)ncell * niso);
  CUDA_OK(cudaMemcpyAsync(d_cell_plane, cell_plane, ncell * 4, cudaMemcpyHostToDevice, s));
  CUDA_OK(cudaMemcpyAsync(d_cell_out, cell_out, ncell * 8, cudaMemcpyHostToDevice, s));
  CellArgs ca;
  ca.cell_plane = d_cell_plane; ca.cell_dens = d_cell_dens; ca.cell_out = d_cell_out;
  ca.plane_T = d_T; ca.plane_base = d_base; ca.cisobeg = d_cisobeg;
  ca.c_idx = w.c_idx.p;
  ca.giown = b->d_giown.p; ca.gidwn = b->d_gidwn.p; ca.gwavn = b->d_gwavn.p;
  ca.S = pa.S; ca.ngroups = std::max<long long>(1, b->ngroups);
  ca.niso = niso; ca.nspec = b->nspec; ca.nout = nout; ca.nwave = b->nwave; ca.osamp = b->osamp;
  ca.nDop = b->nDop; ca.nLor = b->nLor;
  ca.iso_spec = w.iso_spec.p; ca.iso_out = d_iso_out;
  ca.aDop = b->d_aDop.p; ca.aLor = b->d_aLor.p; ca.prof_off = b->d_prof_off.p; ca.prof_size = b->d_prof_size.p;
  ca.pool = b->d_prof.p;
  ca.wn0 = b->wn_lo; ca.own_last = b->wn_lo + (double)(b->nowns - 1) * b->odwn; ca.dwn = b->dwn;
  ca.total_mode = total_mode ? 1 : 0;
  {
    PhaseTimer pt(b, "widths", s);
    widths_kernel<<<ncell, std::max(32, niso), 0, s>>>(ca, cells, w.spec_mass.p, w.spec_radius.p, w.iso_mass.p);
    CUDA_OK(cudaGetLastError());
  }
  {
    PhaseTimer pt(b, "accumulate", s);
    // 512-bin tiles where the grid is fine enough for pressure-broadened profiles to span many
    // tiles; 128-bin tiles otherwise (more CTAs for the small grids)
    int tile = 128;
    if (const char *e = getenv("BART_ACC_TILE")) tile = atoi(e) == 512 ? 512 : atoi(e) == 256 ? 256 : 128;
    int fast = 1;
    if (const char *e = getenv("BART_ACC_FAST")) fast = atoi(e);
    const int ntile = (b->nwave + tile - 1) / tile;
    for (int c0 = 0; c0 < ncell; c0 += 32768) {                  // gridDim.y limit
      const int nc = std::min(32768, ncell - c0);
      CellArgs cb = ca;
      cb.cell_plane += c0; cb.cell_dens += (size_t)c0 * b->nspec; cb.cell_out += c0;
      if (tile == 512) accumulate_kernel<512><<<dim3(ntile, nc), kAccCta, 0, s>>>(cb, cells + (size_t)c0 * niso, d_out, fast);
      else if (tile == 256) accumulate_kernel<256><<<dim3(ntile, nc), kAccCta, 0, s>>>(cb, cells + (size_t)c0 * niso, d_out, fast);
      else accumulate_kernel<128><<<dim3(ntile, nc), kAccCta, 0, s>>>(cb, cells + (size_t)c0 * niso, d_out, fast);
    }
    CUDA_OK(cudaGetLastError());
  }
  CUDA_OK(cudaStreamSynchronize(s));
  long long ne = 0;
  for (int c = 0; c < ncell; c++) ne += total[cell_plane[c]];
  return ne;
}

// planes per batch: bounded by the output buffer (2 GB) -- one plane is nlayer * ngmol * nwave doubles
static int planes_per_batch(const BuilderState *b) {
  const size_t plane_bytes = (size_t)b->nlayer * b->ngmol * b->nwave * 8;
  const size_t by_out = ((size_t)2 << 30) / std::max<size_t>(1, plane_bytes);
  const size_t by_S = ((size_t)8 << 30) / std::max<size_t>(1, (size_t)b->ngroups * 8);   // strengths [plane][group]
  return (int)std::max<size_t>(1, std::min<size_t>(16, std::min(by_out, by_S)));
}

static BuilderState *ensure_builder(BuilderPtr &bp, const Options &o, const Atmosphere &a,
                                    const Molecules &m, Tli &t, const std::vector<double> &wn, cudaStream_t s) {
  if (!bp) bp.reset(new BuilderState());
  BuilderState *b = bp.get();
  if (!t.present) fail("the line-by-line opacity calculation needs a TLI line list (linedb)");
  if (b->nwave == 0) setup_static(b, o, a, m, t, wn);
  build_profiles(b, o, s);
  load_lines(b, o, t, wn, s);
  return b;
}

void builder_slice(BuilderPtr &bp, const Options &o, const Atmosphere &a, const Molecules &m,
                   Tli &t, const std::vector<double> &wn, cudaStream_t s, int t_begin, int t_end,
                   double *host_out) {
  BuilderState *b = ensure_builder(bp, o, a, m, t, wn, s);
  if (!b->grid_ready) setup_grid_temps(b, o, t);
  if (t_begin < 0 || t_end > b->ntemp || t_begin > t_end)
    fail("temperature slice [%d, %d) outside the grid of %d temperatures", t_begin, t_end, b->ntemp);
  const int nt = t_end - t_begin, nl = b->nlayer, ns = b->nspec;
  const size_t plane = (size_t)b->ngmol * b->nwave;
  const int pb = planes_per_batch(b);
  for (int it0 = t_begin; it0 < t_end; it0 += pb) {
    const int np = std::min(pb, t_end - it0), nc = np * nl;
    std::vector<double> pT(np), pZ((size_t)np * b->niso), dens((size_t)nc * ns);
    std::vector<int> cplane(nc);
    std::vector<long long> cout_(nc);
    for (int p = 0; p < np; p++) {
      const int it = it0 + p;
      pT[p] = b->temps[it];
      for (int i = 0; i < b->niso; i++) pZ[(size_t)p * b->niso + i] = b->ziso[(size_t)i * b->ntemp + it];
      // densities: stateeqnford with number abundances (transit.h:58-69, opacity.c:390-394)
      for (int r = 0; r < nl; r++) {
        const int c = p * nl + r;
        cplane[c] = p;
        cout_[c] = (long long)c * (long long)plane;
        for (int j = 0; j < ns; j++) {
          const double rho = kAMU * a.q[(size_t)j * nl + r] * (a.press[r] * a.pfct) / kKB / pT[p];
          dens[(size_t)c * ns + j] = rho * m.mass[j];
        }
      }
    }
    double *d_dens = b->dens.ensure_grow(dens.size());
    double *d_out = b->out.ensure_grow((size_t)nc * plane);
    CUDA_OK(cudaMemcpyAsync(d_dens, dens.data(), dens.size() * 8, cudaMemcpyHostToDevice, s));
    CUDA_OK(cudaMemsetAsync(d_out, 0, (size_t)nc * plane * 8, s));
    b->neval += run_planes(b, o, m, t, np, pT.data(), pZ.data(), nc, cplane.data(), d_dens,
                           cout_.data(), d_out, false, s);
    auto td0 = std::chrono::steady_clock::now();
    // device [plane][layer][mol][wave] -> host [layer][t - t_begin][mol][wave]: one strided copy
    // per plane straight into the caller's buffer (fast when it is pinned, as the file writer's is)
    for (int p = 0; p < np; p++)
      CUDA_OK(cudaMemcpy2DAsync(host_out + (size_t)(it0 + p - t_begin) * plane, (size_t)nt * plane * 8,
                              d_out + (size_t)p * nl * plane, plane * 8, plane * 8, nl,
                              cudaMemcpyDeviceToHost, s));
    CUDA_OK(cudaStreamSynchronize(s));
    b->phase_ms["d2h"] += std::chrono::duration<double, std::milli>(
        std::chrono::steady_clock::now() - td0).count();
  }
}

// Line-by-line forward mode: total molecular extinction (all isotopes collapsed, times the
// species densities) of ncell (model, layer) cells at their own temperatures, written to
// d_out + cell_out[c] (nwave doubles each).  tau.c:163-175,253-264 -> computemolext(permol=0).
void builder_lbl_cells(BuilderPtr &bp, const Options &o, const Atmosphere &a, const Molecules &m,
                       Tli &t, const std::vector<double> &wn, cudaStream_t s, int ncell,
                       const double *cell_T, const double *d_cell_dens, const long long *cell_out,
                       double *d_out) {
  BuilderState *b = ensure_builder(bp, o, a, m, t, wn, s);
  if (b->zspline.empty()) {                 // second derivatives of Z_iso(T), makesample.c:534-544
    b->zspline.resize(b->niso);
    for (int i = 0; i < b->niso; i++) {
      const std::vector<double> &T = t.db[t.iso_db[i]].T;
      b->zspline[i].resize(T.size());
      spline_second_derivs(T.data(), t.iso_Z[i].data(), (long)T.size(), b->zspline[i].data());
    }
  }
  // bound the per-batch work arrays: block counters are nblk ints per plane
  const long long nblk = std::max<long long>(1, (b->ngroups + kCompactThreads - 1) / kCompactThreads);
  const long long by_S = ((long long)8 << 30) / std::max<long long>(1, b->ngroups * 8);     // strengths [plane][group]
  const int maxp = (int)std::max<long long>(1, std::min<long long>(std::min<long long>(16384, by_S), ((long long)1 << 28) / nblk));
  std::vector<int> cplane;
  std::vector<double> pZ;
  for (int c0 = 0; c0 < ncell; c0 += maxp) {
    const int nc = std::min(maxp, ncell - c0);
    cplane.resize(nc); pZ.resize((size_t)nc * b->niso);
    for (int c = 0; c < nc; c++) {
      cplane[c] = c;
      for (int i = 0; i < b->niso; i++) {
        const std::vector<double> &T = t.db[t.iso_db[i]].T;
        pZ[(size_t)c * b->niso + i] = spline_eval(b->zspline[i].data(), (long)T.size(), T.data(),
                                                  t.iso_Z[i].data(), cell_T[c0 + c]);
      }
    }
    b->neval += run_planes(b, o, m, t, nc, cell_T + c0, pZ.data(), nc, cplane.data(),
                           d_cell_dens + (size_t)c0 * b->nspec, cell_out + c0, d_out, true, s);
  }
}

void builder_run_and_write(BuilderPtr &bp, const Options &o, const Atmosphere &a,
                           const Molecules &m, Tli &t, const std::vector<double> &wn,
                           cudaStream_t s, const std::string &path) {
  BuilderState *b = ensure_builder(bp, o, a, m, t, wn, s);
  if (!b->grid_ready) setup_grid_temps(b, o, t);
  OpacityGrid g;
  g.nmol = b->ngmol; g.ntemp = b->ntemp; g.nlayer = b->nlayer; g.nwave = b->nwave;
  g.molid = b->gmol_id; g.temp = b->temps; g.wn = wn;
  g.press.resize(b->nlayer);
  // opacity.c:344-346.  The reference stores the pressures after its identity spline resample
  // (makesample.c:507-531, compiled -ffast-math): the top layer differs by ~1 ulp from the file value.
  for (int r = 0; r < b->nlayer; r++) g.press[r] = a.press[r] * a.pfct;
  // $BART_TSLICE="begin:end" builds only a slice of the temperature axis and writes its planes
  // in place (one process per GPU shards the axis; rank 0 writes the header first)
  int t0 = 0, t1 = b->ntemp;
  bool header = true;
  // Honoured only under --justOpacity: a leftover variable in the environment of a normal run whose
  // opacity file is missing must not leave a file with one temperature slice filled in.
  if (const char *e = o.justOpacity ? getenv("BART_TSLICE") : nullptr) {
    if (sscanf(e, "%d:%d", &t0, &t1) != 2) fail("BART_TSLICE must be 'begin:end'");
    if (t0 < 0 || t1 < t0 || t1 > b->ntemp)
      fail("BART_TSLICE %d:%d is outside the temperature axis [0, %d]", t0, t1, b->ntemp);
    header = t0 == 0;
  }
  const size_t plane = (size_t)b->ngmol * b->nwave;
  // Streaming writer: the planes of a batch of temperatures are built, copied back and written in
  // place (file order o[layer][temp][mol][wave], opacity.c:418-421), so host memory holds one
  // batch (<= 2 GB) however large the grid is.  Rank 0 / the first slice writes the header.
  const Fd fd(path.c_str(), O_WRONLY | O_CREAT | (t0 == 0 && t1 == b->ntemp ? O_TRUNC : 0), 0644);
  if (fd < 0) fail("Opacity filename '%s' cannot be opened for writing.", path.c_str());
  const long long hdr = 4 * sizeof(long) + g.nmol * sizeof(int) + (g.ntemp + g.nlayer + g.nwave) * 8;
  // every slice writer sets the file to its final size: a stale, larger file of other dimensions
  // does not survive, and the slices can be written in any order
  if (ftruncate(fd, hdr + (long long)g.nlayer * g.ntemp * (long long)plane * 8) != 0)
    fail("Opacity filename '%s' cannot be sized.", path.c_str());
  if (header) {
    std::vector<char> h(hdr);
    char *p = h.data();
    long dims[4] = {g.nmol, g.ntemp, g.nlayer, g.nwave};
    memcpy(p, dims, sizeof(dims)); p += sizeof(dims);
    memcpy(p, g.molid.data(), g.nmol * sizeof(int)); p += g.nmol * sizeof(int);
    memcpy(p, g.temp.data(), g.ntemp * 8); p += g.ntemp * 8;
    memcpy(p, g.press.data(), g.nlayer * 8); p += g.nlayer * 8;
    memcpy(p, g.wn.data(), g.nwave * 8);
    if (pwrite(fd, h.data(), hdr, 0) != hdr) fail("short write on '%s'", path.c_str());
  }
  const int pb = planes_per_batch(b);
  PinnedBuf<double> slab;                                   // pinned staging for one batch
  if (t1 > t0) slab.ensure((size_t)b->nlayer * std::min(pb, t1 - t0) * plane);
  for (int it0 = t0; it0 < t1; it0 += pb) {
    const int nt = std::min(pb, t1 - it0);
    builder_slice(bp, o, a, m, t, wn, s, it0, it0 + nt, slab.p);
    auto tw0 = std::chrono::steady_clock::now();
    for (int r = 0; r < b->nlayer; r++) {
      const long long off = hdr + ((long long)r * g.ntemp + it0) * (long long)plane * 8;
      const long long len = (long long)nt * plane * 8;
      const char *src = (const char *)(slab.p + (size_t)r * nt * plane);
      for (long long done = 0; done < len;) {               // pwrite may be partial above 2 GB
        const ssize_t w = pwrite(fd, src + done, (size_t)std::min<long long>(len - done, 1LL << 30), off + done);
        if (w <= 0) fail("short write on '%s'", path.c_str());
        done += w;
      }
    }
    b->phase_ms["file_write"] += std::chrono::duration<double, std::milli>(
        std::chrono::steady_clock::now() - tw0).count();
  }
}

long long builder_stats(BuilderState *b, long long *nlines, long long *ngroups, long long *neval) {
  if (!b) return -1;
  if (nlines) *nlines = b->nlines;
  if (ngroups) *ngroups = b->ngroups;
  if (neval) *neval = b->neval;
  return b->nlines;
}

double builder_phase_ms(BuilderState *b, const char *name) {
  if (!b) return -1.0;
  auto it = b->phase_ms.find(name);
  return it == b->phase_ms.end() ? 0.0 : it->second;
}

long long builder_line_bins(BuilderState *b, long long *iown_out, long long capacity) {
  if (b->h_iown.empty() && b->d_trace.p && b->nlines > 0) {
    b->h_iown.resize((size_t)b->nlines);
    CUDA_OK(cudaMemcpy(b->h_iown.data(), b->d_trace.p, (size_t)b->nlines * 4, cudaMemcpyDeviceToHost));
  }
  const long long n = (long long)b->h_iown.size();
  for (long long i = 0; i < n && i < capacity; i++) iown_out[i] = b->h_iown[i];
  return n;
}

int builder_profile(BuilderState *b, int idop, int ilor, float *out, long long capacity,
                    long long *halfsize) {
  if (!b->profiles_ready) fail("Voigt profiles have not been computed");
  if (idop < 0 || idop >= b->nDop || ilor < 0 || ilor >= b->nLor) fail("profile index out of range");
  const size_t p = (size_t)idop * b->nLor + ilor;
  const long long n = 2 * b->prof_size[p] + 1;
  if (halfsize) *halfsize = b->prof_size[p];
  if (out) {
    if (capacity < n) fail("profile buffer too small (%lld needed)", n);
    const long long K = (n - 1) / b->osamp + 1;
    std::vector<float> tr((size_t)b->osamp * K);
    CUDA_OK(cudaMemcpy(tr.data(), b->d_prof.p + b->prof_off[p], tr.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (long long i = 0; i < n; i++) out[i] = tr[(size_t)(i % b->osamp) * K + i / b->osamp];
  }
  return 0;
}

void builder_free(BuilderState *b) { delete b; }

}  // namespace bart
