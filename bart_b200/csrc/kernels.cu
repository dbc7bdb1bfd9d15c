// kernels.cu -- sm_100a kernels of the forward model (stages a, b, c of the north star).
//
//   atm_prep_kernel        K0   one CTA per model: densities, hydrostatic radii, per-layer tables
//   eclipse_column_kernel  K1+K2e+K3e fused: opacity lookup + tau scan + intensity + flux
//   transit_weights_kernel K2t  chord-integration weights per model
//   transit_column_kernel  K1+K2t+K3t fused: lookup + chord tau + modulation
//   extinction_kernel      K1 stand-alone lookup (materialises extinction; roofline/debug)
//   band_integrate_kernel  K4   batched fp64 filter-band reduction
//
// Thread mapping: thread <-> wavenumber (the grid's contiguous axis), sequential over depth, so
// every global load of the opacity grid is a fully coalesced 256-byte-per-warp stream and the
// tau scan needs no cross-thread communication.  The per-model coefficient table (~18 KB) is
// staged into shared memory with ONE bulk-async (TMA) copy per CTA and read as warp-wide
// broadcasts.  CTAs are ordered model-fastest inside a wavenumber tile so that concurrently
// resident CTAs stream the same grid columns (different temperature planes) through the L2.
// Tensor cores are not used: nothing here is a dense contraction (4 flop per 16 B).
#include "column_math.cuh"
#include "kernels.hpp"
#include "dyn_smem.hpp"
#include <cuda_runtime.h>
#include <cstring>
#include <cstdlib>
#include <algorithm>
#include <type_traits>

namespace bart {

// ---------------------------------------------------------------------------------------
// TMA bulk copy (cp.async.bulk, SASS UBLKCP) + mbarrier helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// arrive (release.cta): what the arriving thread wrote -- and, after a __syncwarp, what its warp
// wrote -- is visible to a thread whose try_wait (acquire.cta) sees the phase complete
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!ok);
}

// Stage one model's table into shared memory.  Bulk-async when the size allows (multiple of 16 B,
// always true by TabLayout::stride), else a cooperative copy.
// exp table entries (column_math.cuh exp_table_entry; then one weighted copy per ray angle,
// fill_ecl_exp_table) in global memory, copied to shared per CTA
__device__ unsigned long long g_exp_table[(1 + kMaxAng) * kExpTabSize];

__device__ __forceinline__ void stage_table(double *s_tab, const double *g_tab, int ndoubles,
                                            uint64_t *bar, bool use_tma,
                                            unsigned long long *s_etab = nullptr,
                                            int n_etab = kExpTabSize) {
  if (s_etab)
    for (int j = threadIdx.x; j < n_etab; j += blockDim.x) s_etab[j] = g_exp_table[j];
  if (use_tma) {
    if (threadIdx.x == 0) { mbar_init(bar, 1); fence_mbar_init(); }
    __syncthreads();
    if (threadIdx.x == 0) {
      const uint32_t bytes = (uint32_t)ndoubles * 8u;
      mbar_expect_tx(bar, bytes);
      // bulk copies are limited by the mbarrier tx-count (2^20-1); chunk for safety
      uint32_t off = 0;
      while (off < bytes) {
        uint32_t n = bytes - off;
        if (n > 65536u) n = 65536u;
        bulk_g2s((char *)s_tab + off, (const char *)g_tab + off, n, bar);
        off += n;
      }
    }
    mbar_wait(bar, 0);
    if (s_etab) __syncthreads();               // the exp table is written by a generic-proxy store
  } else {
    for (int i = threadIdx.x; i < ndoubles; i += blockDim.x) s_tab[i] = g_tab[i];
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------
// K0
// Everything a model's preparation reads more than once -- its profile, the pressure / mass /
// polarizability columns and the temperature axes the bracket searches walk (opacity grid, CIA
// tables) -- is staged into shared memory by one round of coalesced loads, and the record table is
// assembled there and written out as one coalesced stream: at MC3's population sizes (3-10 models per
// launch) this kernel is a chain of memory latencies, not of arithmetic (a binary search over a
// global array alone is five dependent ~0.3 us round trips).  Same arithmetic, same order.
constexpr int kPrepThreads = 256;
__host__ __device__ inline size_t atm_prep_smem_doubles(const DevConfig &c) {
  size_t n = ((size_t)c.nspec + 3) * c.nlayer;                 // rho, mu, radius, hydrostatic coefficients
  n += ((size_t)c.nspec + 1) * c.nlayer;                       // the model's profile
  n += (size_t)c.nlayer + c.ntemp + 2 * (size_t)c.nspec;       // press, gtemp, mass, pol
  for (int f = 0; f < c.ncia; f++) n += c.cia_nt[f];
  n += (size_t)c.lay.stride();                                 // the record table
  return n + 8;
}
__global__ void __launch_bounds__(kPrepThreads)
atm_prep_kernel(DevConfig c, Knobs knobs, const double *__restrict__ profiles, int n_in,
                double *__restrict__ tabs, int *__restrict__ status,
                const int *__restrict__ pre_status, int nmodels, int staged) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int m = blockIdx.x;
  if (m >= nmodels) return;
  if (pre_status && pre_status[m] != 0) {        // rejected by the input converter already
    if (threadIdx.x == 0) status[m] = pre_status[m];
    return;
  }
  const int nl = c.nlayer;
  double *s_rho = reinterpret_cast<double *>(smem_raw);        // [nspec][nl]
  double *s_mu = s_rho + (size_t)c.nspec * nl;                 // [nl]
  double *s_rad = s_mu + nl;                                   // [nl]
  double *s_hc = s_rad + nl;                                   // [nl]
  __shared__ int s_status;
  if (threadIdx.x == 0) s_status = 0;
  const double *in = profiles + (size_t)m * n_in;
  double *tab = tabs + (size_t)m * c.lay.stride();
  const double *s_in = in;                                     // unstaged (very large configurations):
  double *s_tabrec = tab;                                      // everything straight from / to HBM
  PrepPtrs pp = prep_ptrs_of(c);
  if (staged) {
    double *w_in = s_hc + nl;                                  // [(1 + nspec)][nl]
    double *s_press = w_in + ((size_t)c.nspec + 1) * nl;       // [nl]
    double *s_gtemp = s_press + nl;                            // [ntemp]
    double *s_mass = s_gtemp + c.ntemp;                        // [nspec]
    double *s_pol = s_mass + c.nspec;                          // [nspec]
    double *s_ciaT = s_pol + c.nspec;                          // [sum cia_nt]
    const int nprof = (c.nspec + 1) * nl;
    for (int i = threadIdx.x; i < nprof; i += blockDim.x) w_in[i] = in[i];
    for (int i = threadIdx.x; i < nl; i += blockDim.x) s_press[i] = c.press[i];
    for (int i = threadIdx.x; i < c.ntemp; i += blockDim.x) s_gtemp[i] = c.gtemp[i];
    for (int i = threadIdx.x; i < c.nspec; i += blockDim.x) { s_mass[i] = c.mass[i]; s_pol[i] = c.pol ? c.pol[i] : 0.0; }
    double *dst = s_ciaT;
#pragma unroll
    for (int f = 0; f < kMaxCia; f++)
      if (f < c.ncia) {
        for (int i = threadIdx.x; i < c.cia_nt[f]; i += blockDim.x) dst[i] = c.ciaT[f][i];
        pp.ciaT[f] = dst;
        dst += c.cia_nt[f];
      }
    pp.press = s_press; pp.gtemp = s_gtemp; pp.mass = s_mass; pp.pol = s_pol;
    s_in = w_in;
    s_tabrec = dst + ((reinterpret_cast<uintptr_t>(dst) & 8) ? 1 : 0);   // 16-byte aligned records
  }
  __syncthreads();
  // The stages are dealt out so that no thread carries a long dependent chain (at 3-10 models per
  // launch the kernel's time is its longest chain): densities per (species, layer) pair; the record
  // parts that do not need the radii (thermal / CIA / scattering, one part per thread) run on the other
  // warps while thread 0 walks the hydrostatic recurrence.
  int st = 0;
  for (int i = threadIdx.x; i < c.nspec * nl; i += blockDim.x) {
    const int j = i / nl, l = i - j * nl;
    s_rho[i] = prep_density(c, pp, s_in, l, j);
  }
  for (int l = threadIdx.x; l < nl; l += blockDim.x) st |= prep_mu(c, pp, s_in, l, s_mu + l);
  __syncthreads();
  const KnobVals kv = knobs_for(knobs, m);
  for (int l = threadIdx.x; l < nl - 1; l += blockDim.x) s_hc[l] = hydro_coef(c, pp, s_in, s_mu, l);
  __syncthreads();
  if (knobs.radius_file) {
    for (int l = threadIdx.x; l < nl; l += blockDim.x) s_rad[l] = knobs.radius_file[l];
  } else if (threadIdx.x == 0 || threadIdx.x == 32)          // one direction each, in different warps
    hydrostatic_radii(c, pp, kv.r0, s_in, s_mu, s_hc, s_rad, threadIdx.x == 0 ? 1 : 2);
  {
    // warps 0 and 1 are busy with the radii unless they come from the file
    const int first = knobs.radius_file ? 0 : 64;
    const int nthr = (int)blockDim.x - first;
    if ((int)threadIdx.x >= first)
      for (int i = (int)threadIdx.x - first; i < 3 * nl; i += nthr) {
        const int part = i / nl, d = i - part * nl;
        if (part == 0) st |= prep_row_thermal(c, pp, d, s_in, s_rho, nl, s_tabrec, c.lbl_model0 + m);
        else if (part == 1) st |= prep_row_cia(c, pp, d, s_in, s_rho, nl, s_tabrec);
        else prep_row_scat(c, pp, kv, d, s_in, s_rho, nl, s_tabrec);
      }
  }
  __syncthreads();
  for (int d = threadIdx.x; d < nl; d += blockDim.x) prep_row_radius(c, d, s_rad, s_tabrec);
  if (c.lbl)
    for (int i = threadIdx.x; i < nl * c.nspec; i += blockDim.x) {
      const int l = i / c.nspec, j = i - l * c.nspec;
      c.lbl_dens[((size_t)(c.lbl_model0 + m) * nl + l) * c.nspec + j] = s_rho[(size_t)j * nl + l];
    }
  if (st) atomicOr(&s_status, st);
  __syncthreads();
  if (staged) {
    const int nd = c.lay.stride();
    for (int i = threadIdx.x; i < nd; i += blockDim.x) tab[i] = s_tabrec[i];
  }
  if (threadIdx.x == 0) status[m] = s_status;
}

// ---------------------------------------------------------------------------------------
// fused eclipse column kernel
// Specialised builds with at most one CIA file: 96 registers, 10 CTAs (20 warps) per SM, no spills --
// each depth step loads its own grid and CIA samples (eclipse_columns with AHEAD false), so they are not
// live across D(tau).  W12, 4096 models, B200 at 1000 W (profiles/r03_eclipse_column_variants.json):
// 3.77 ms against 4.12 ms for the former one-depth-ahead prefetch at 128 registers / 16 warps (12 bytes
// spilled).  Measured alternatives: the same in-step loads at 128 registers / 16 warps 3.94 ms; the lo
// plane one depth ahead at 96 registers 4.03 ms and the loads issued at the end of the previous step
// 4.06 ms (both spill 8 bytes).  Before that: 112 registers / 18 warps 4.43 ms (spills go through the
// L1 data pipe, the busiest unit), 144 registers / 14 warps 5.07 ms.  Two CIA files, the run-time-count
// and the introspection builds keep 8 CTAs (the two-CIA builds spill at 96).  One column per thread (the slot kernel's
// arithmetic) in CTAs of 128 threads at 72 registers, 28 warps per SM: 4.30 against 4.12 ms -- the
// depth's table record is then read per column and the Planck chaining is lost.
template <int NMOL, int NCIA, int NANG, bool KEEP, int SQ, bool SC, bool AHEAD>
__global__ void __launch_bounds__(kEclThreads, CellData<NMOL, NCIA>::kStaticCia && NCIA <= 1 && !KEEP && !AHEAD ? 10 : 8)
eclipse_column_kernel(DevConfig c, const double *__restrict__ tabs, const int *__restrict__ status,
                      double *__restrict__ spectra, double *__restrict__ tau_keep,
                      int *__restrict__ last_keep, int nmodels, int use_tma) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  // exp tables (plain + one per ray angle), one 128-byte bank row each
  unsigned long long *s_etab = reinterpret_cast<unsigned long long *>(smem_raw);
  const int n_etab = ecl_tab_entries(NANG > 0 ? NANG : c.nang);
  double *s_tab = reinterpret_cast<double *>(s_etab + n_etab);
  const int m = blockIdx.x % nmodels;           // model-fastest: neighbours share grid columns
  const int tile = blockIdx.x / nmodels;
  const int w0 = tile * (kEclThreads * kEclCols) + threadIdx.x;
  const int nd = c.lay.stride();
  double *out = spectra + (size_t)m * c.nwave;
  if (status[m] != 0) {                          // rejected model: -1 fill (BARTfunc.py:327-330)
#pragma unroll
    for (int k = 0; k < kEclCols; k++)
      if (w0 + k * kEclThreads < c.nwave) out[w0 + k * kEclThreads] = -1.0;
    return;
  }
  stage_table(s_tab, tabs + (size_t)m * nd, nd, &bar, use_tma != 0, s_etab, n_etab);
  // thread t carries columns w0 and w0 + 64: each is its own coalesced stream, addressed from one
  // base pointer with compile-time offsets.  Columns past the end of the spectrum idle (the warp
  // votes need all lanes); their loads land in the padding behind the grid and the CIA tables.
  bool valid[kEclCols];
  double *tk[kEclCols];
  int *lk[kEclCols];
  double flux[kEclCols];
#pragma unroll
  for (int k = 0; k < kEclCols; k++) {
    const int wk = w0 + k * kEclThreads;
    valid[k] = wk < c.nwave;
    const int wc = min(wk, c.nwave - 1);
    tk[k] = KEEP ? tau_keep + ((size_t)m * c.nwave + wc) * c.nlayer : nullptr;
    lk[k] = KEEP ? last_keep + (size_t)m * c.nwave + wc : nullptr;
  }
  // the specialised instantiations leave the Planck-exponent clamp out and evaluate the Planck
  // exponential to degree 4 (launch_eclipse routes configurations that need more to the
  // run-time-count kernel)
  eclipse_columns<NMOL, NCIA, NANG, KEEP, kEclCols, SQ, true, kEclThreads, NMOL == 0, SC, AHEAD>(
      c, s_tab, s_etab, w0, valid, tk, lk, flux);
#pragma unroll
  for (int k = 0; k < kEclCols; k++)
    if (valid[k]) out[w0 + k * kEclThreads] = flux[k];
}

// Small batches (BART's own populations are ~10 chains): CTA = one warp = one slot of 32
// consecutive columns of one model, one column per thread -- four times the CTAs of the kernel
// above, each with a quarter of its work, so that a 10-model generation spreads over the whole
// machine instead of occupying ~190 CTAs for 100 dependent depth steps.  Same column arithmetic
// (eclipse_columns with NCOL 1; `upper` chains the Planck exponential exactly like the second
// column of a thread above), so spectra are bit-identical whichever kernel a batch size selects.
template <int NMOL, int NCIA, int NANG, int SQ, bool SC>
__global__ void __launch_bounds__(32)
eclipse_slot_kernel(DevConfig c, const double *__restrict__ tabs, const int *__restrict__ status,
                    double *__restrict__ spectra, int nmodels, int use_tma) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  unsigned long long *s_etab = reinterpret_cast<unsigned long long *>(smem_raw);
  const int n_etab = ecl_tab_entries(NANG > 0 ? NANG : c.nang);
  double *s_tab = reinterpret_cast<double *>(s_etab + n_etab);
  const int m = blockIdx.x % nmodels;
  const int slot = blockIdx.x / nmodels;
  const int w = slot * 32 + threadIdx.x;
  const int nd = c.lay.stride();
  double *out = spectra + (size_t)m * c.nwave;
  if (status[m] != 0) {
    if (w < c.nwave) out[w] = -1.0;
    return;
  }
  stage_table(s_tab, tabs + (size_t)m * nd, nd, &bar, use_tma != 0, s_etab, n_etab);
  // the slot's place in the 128-column tile of eclipse_column_kernel: second half = a thread's
  // second column there
  const bool upper = c.planck_cols > 0 && ((slot * 32) % (kEclThreads * kEclCols)) >= kEclThreads;
  const bool valid[1] = {w < c.nwave};
  double *tk[1] = {nullptr};
  int *lk[1] = {nullptr};
  double flux[1];
  eclipse_columns<NMOL, NCIA, NANG, false, 1, SQ, true, kEclThreads, NMOL == 0, SC>(c, s_tab, s_etab, w, valid, tk,
                                                                                    lk, flux, upper);
  if (valid[0]) out[w] = flux[0];
}

// Latency kernel for the smallest batches (one run_transit call, a 3-10 chain MC3 generation):
// lanes <-> LAYERS.  A warp owns kScanCols adjacent wavenumber columns of one model at a time;
// lane = (depth in round) * kScanCols + column, so one round covers 32 / kScanCols = 8 consecutive
// depths of 4 columns, and the lookups, Planck functions and D(tau) of those depths proceed side by
// side instead of as dependent steps of one thread (100 layers: 13 rounds instead of 100 steps):
//   extinction  a lane reads ITS depth's table record (the four lanes of a depth broadcast) and its
//               two 32-byte grid samples + one per CIA file; the four columns of a depth are
//               contiguous in the grid, so a warp's load touches 8 full 128-byte lines like the
//               throughput kernel's (lanes <-> 32 layers of ONE column measured 7 us per model: 32
//               lines of one sector each per load);
//   tau         top-aligned Simpson prefix (eclipse_columns above): the panel that ends at an even
//               depth d is SA er[d] + SB er[d-1] + SC er[d-2] (neighbours by shuffle, the previous
//               round's last two depths carried), tau(even d) = inclusive segmented scan of the
//               panels over the round + carry, tau(odd d) = tau(d-1) + TR (er[d] + er[d-1]);
//   last        first depth with tau > toomuch: ballot + find-first-set per column; a finished
//               column idles and the warp leaves when its four columns are done;
//   flux        trapezoid terms (D_d - D_{d-1})(B_d + B_{d-1}) for 1 <= d <= last summed per lane
//               over the rounds, one butterfly reduction per column at the end.
// The panels are summed in scan order, the series / exponentials choice for D(tau) is taken per lane
// and the Planck exponential is not chained between columns: spectra agree with the throughput
// kernel to the accuracy of those approximations (~1e-11 relative), not to the bit.  Configurations
// outside the specialised instantiations (run-time molecule / CIA counts, the per-column Planck
// clamp) stay on the slot kernel.
constexpr int kScanThreads = 128;                // 4 warps: fine-grained CTAs balance a 10-model batch over the SMs
constexpr int kScanCols = 4;                     // columns per warp task
constexpr int kScanDepths = 32 / kScanCols;      // depths per round
constexpr long long kScanMaxColumns = 40000;     // batches up to this many (model, wavenumber) columns take it
template <int NMOL, int NCIA, int NANG, int SQ, bool SC>
__device__ __forceinline__ double eclipse_scan_columns(const DevConfig &c, const double *tab,
                                                       const unsigned long long *etab, int w0, int lane) {
  typedef TabLayout L;
  const unsigned FULL = 0xffffffffu;
  const int nl = c.nlayer, nf = c.lay.nf();
  const int nang = NANG > 0 ? NANG : c.nang;
  const int small_hi = hi_word(c.tau_small);
  const int col = lane & (kScanCols - 1), dl = lane / kScanCols;
  const int w = min(w0 + col, c.nwave - 1);                    // a column past the end repeats the last one
  const double wn = c.wn[w];
  const double wn4 = (wn * wn) * (wn * wn);
  const double c2n = cH * wn * cLS / cKB * kExpScale;          // Planck exponent x N/ln2, per 1/T
  const ColPtrs P = col_ptrs<NCIA>(c, w);
  const bool odd = dl & 1;                                     // rounds start at even depths
  const int top = (kScanDepths - 1) * kScanCols + col;         // lane of the round's last depth, this column
  double s_carry = 0.0;                                        // Simpson sum at the end of the previous round
  double er_p = 0.0, d_p = c.d0, b_p = 0.0;                    // this lane's er, D, B of the previous round
  double trap = 0.0, BL = 0.0, DL = 0.0;
  bool done = false;                                           // this lane's column has its `last`
  const int nround = (nl + kScanDepths - 1) / kScanDepths;
  CellData<NMOL, NCIA> x;
  cell_load<NMOL, NCIA>(c, P, tab + (size_t)min(dl, nl - 1) * nf, x);
  for (int r = 0; r < nround; r++) {
    const int d = r * kScanDepths + dl;
    const bool live = d < nl;
    const double *row = tab + (size_t)(live ? d : nl - 1) * nf;
    const double er = cell_combine<NMOL, NCIA, SC>(c, P, row, x, wn4, 0);
    // the next round's samples (same registers) are in flight under the rest of this round
    cell_load<NMOL, NCIA>(c, P, tab + (size_t)min(d + kScanDepths, nl - 1) * nf, x);
    // Planck function without its prefactor (eclipse_intens, eclipse.c:130-140)
    const double B = fast_rcp1(exp_w(c2n, row[L::INVT], etab, -1.0));
    const D2 s1 = ld2(row + L::SA);                             // (SA, SB)
    const D2 s2 = ld2(row + L::SC);                             // (SC, TR)
    // er of the two depths above by lane rotation: the lanes of the round's last two depths hand over
    // what they held in the previous round (depths 8 r - 1, 8 r - 2)
    const double e1 = __shfl_sync(FULL, dl == kScanDepths - 1 ? er_p : er, (lane - kScanCols) & 31);
    const double e2 = __shfl_sync(FULL, dl >= kScanDepths - 2 ? er_p : er, (lane - 2 * kScanCols) & 31);
    double v = (!odd && d >= 2 && live) ? fma(s1.x, er, fma(s1.y, e1, s2.x * e2)) : 0.0;
#pragma unroll
    for (int s = 1; s < kScanDepths; s <<= 1) {
      const double t = __shfl_up_sync(FULL, v, s * kScanCols);
      if (dl >= s) v += t;
    }
    const double S = s_carry + v;                               // Simpson sum up to the last even depth <= d
    double tau = odd ? fma(s2.y, er + e1, S) : S;
    if (d == 0) tau = 0.0;
    const bool cross = !done && live && (d >= 1 ? tau > c.toomuch : 0.0 > c.toomuch);
    const unsigned bal = (__ballot_sync(FULL, cross) >> col) & 0x11111111u;   // this column's depths
    const int first = bal ? (__ffs(bal) - 1) / kScanCols : kScanDepths;       // depth-in-round of `last`
    const bool use = !done && live && d >= 1 && dl <= first;    // depths 1..last enter the flux
    double D = c.d0;
    if (use) {
      if (hi_word(tau) < small_hi) {
        const double u = fma(tau, c.ser_s, -1.0);
        double p = c.taylor[kTaylorN - 1];
#pragma unroll
        for (int i = kTaylorN - 2; i >= 0; i--) p = fma(p, u, c.taylor[i]);
        D = p;
      } else {
        const double tc = tau < c.tau_clamp ? tau : c.tau_clamp;   // exp arguments stay above -690
        if (SQ >= 0) {
          const double e = exp_w(tc, -c.exp_a[SQ >> 4], etab + (1 + (SQ >> 4)) * kExpTabSize, 0.0);
          D = fma(e * e, c.sq_coef, e);
        } else D = 0.0;
#pragma unroll
        for (int a = 0; a < (NANG > 0 ? NANG : kMaxAng); a++)
          if (a < nang && !(SQ >= 0 && (a == (SQ >> 4) || a == (SQ & 15))))
            D = exp_w(tc, -c.exp_a[a], etab + (1 + a) * kExpTabSize, D);
      }
    }
    const double Dm = __shfl_sync(FULL, dl == kScanDepths - 1 ? d_p : D, (lane - kScanCols) & 31);
    const double Bm = __shfl_sync(FULL, dl == kScanDepths - 1 ? b_p : B, (lane - kScanCols) & 31);
    if (use) trap = fma(D - Dm, B + Bm, trap);
    // the column's last depth: the crossing, or the bottom layer in the final round
    const bool ends = !done && (bal != 0u || r == nround - 1);
    const int f = (bal ? first : (nl - 1) % kScanDepths) * kScanCols + col;
    const double bf = __shfl_sync(FULL, B, f), df = __shfl_sync(FULL, D, f);
    if (ends) { BL = bf; DL = df; done = true; }
    if (__all_sync(FULL, done)) break;
    s_carry += __shfl_sync(FULL, v, top);
    er_p = er; d_p = D; b_p = B;
  }
#pragma unroll
  for (int s = 16; s >= kScanCols; s >>= 1) trap += __shfl_xor_sync(FULL, trap, s);
  const double c1 = 2.0 * cH * (wn * wn * wn) * cLS * cLS;
  return cPI * c1 * (BL * DL - 0.5 * trap);                     // lanes 0 .. kScanCols-1 hold their column's flux
}

template <int NMOL, int NCIA, int NANG, int SQ, bool SC>
__global__ void __launch_bounds__(kScanThreads, 6)
eclipse_scan_kernel(DevConfig c, const double *__restrict__ tabs, const int *__restrict__ status,
                    double *__restrict__ spectra, int nmodels, int use_tma, int tasks_per_warp) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  unsigned long long *s_etab = reinterpret_cast<unsigned long long *>(smem_raw);
  const int n_etab = ecl_tab_entries(NANG > 0 ? NANG : c.nang);
  double *s_tab = reinterpret_cast<double *>(s_etab + n_etab);
  constexpr int kWarps = kScanThreads / 32;
  const int m = blockIdx.x % nmodels;
  const int tile = blockIdx.x / nmodels;
  const int per = kWarps * tasks_per_warp * kScanCols;         // columns of one CTA
  const int wbase = tile * per;
  const int nd = c.lay.stride();
  double *out = spectra + (size_t)m * c.nwave;
  if (status[m] != 0) {                          // rejected model: -1 fill (BARTfunc.py:327-330)
    for (int i = threadIdx.x; i < per; i += blockDim.x)
      if (wbase + i < c.nwave) out[wbase + i] = -1.0;
    return;
  }
  stage_table(s_tab, tabs + (size_t)m * nd, nd, &bar, use_tma != 0, s_etab, n_etab);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // the warps of a CTA work on adjacent column groups at the same time
  for (int j = 0; j < tasks_per_warp; j++) {
    const int w0 = wbase + (j * kWarps + warp) * kScanCols;
    if (w0 >= c.nwave) break;
    const double flux = eclipse_scan_columns<NMOL, NCIA, NANG, SQ, SC>(c, s_tab, s_etab, w0, lane);
    if (lane < kScanCols && w0 + lane < c.nwave) out[w0 + lane] = flux;
  }
}

// ---------------------------------------------------------------------------------------
// transit geometry
//
// transit_weights_kernel: one CTA per model; writes the chord weights in the tiled layout of
// column_math.cuh (zero-filled first: weights above the diagonal are zero).  kTwParts threads share
// a depth's row (contiguous shares of its Simpson panels), the radii come from shared memory and
// every weight is stored once: the first form -- a thread per depth adding each panel's terms into
// global memory -- was a chain of ~150 dependent read-modify-write round trips, 51 us per launch
// whatever the batch size.
constexpr int kTwParts = 4, kTwThreads = 512;   // (8 x 1024: 13.8 vs 15.9 us small, 0.23 vs 0.18 ms per 4096 models)
__global__ void __launch_bounds__(kTwThreads)
transit_weights_kernel(DevConfig c, const double *__restrict__ tabs, double *__restrict__ wts,
                       int nmodels, int mma_layout, int *__restrict__ status_col) {
  extern __shared__ double s_radius[];          // [nlayer] radii by depth
  const int m = blockIdx.x;
  if (m >= nmodels) return;
  if (status_col && threadIdx.x == 0) status_col[m] = 0;      // (saves the launch a memset node)
  const int nl = c.nlayer, nf = c.lay.nf();
  const size_t stride = mma_layout ? mm_stride(nl) : tr_stride(nl);
  const double *tab = tabs + (size_t)m * c.lay.stride();
  double *wm = wts + (size_t)m * stride;
  for (int i = threadIdx.x; i < nl; i += blockDim.x) s_radius[i] = tab[(size_t)i * nf + TabLayout::RAD];
  for (size_t i = threadIdx.x; i < stride; i += blockDim.x) wm[i] = 0.0;
  __syncthreads();
  for (int item = threadIdx.x; item < nl * kTwParts; item += blockDim.x) {
    const int d = item / kTwParts, part = item - d * kTwParts;
    if (mma_layout) transit_weight_row_mm(c, s_radius, d, wm, part, kTwParts);
    else transit_weight_row_tiled(c, s_radius, d, wm, part, kTwParts);
  }
}

// transit_tile_kernel: CTA = one model x 64 wavenumbers, 4 warps.  The chord optical depth
// tau(d, w) = sum_{i<=d} W[d][i] er[i][w] (totaltau1, slantpath.c:18-108) is a triangular
// matrix product per model; it is evaluated in depth chunks of kTrChunk with a register tile
// (lane: 2 wavenumbers x 5 depths; warp: 64 wavenumbers x 5 depths; CTA: the chunk's 20 depths):
//   phase A  all threads: opacity lookup of the chunk's 20 layers -> er[layer][64] in shared memory
//   phase B  tau of the chunk: er rows as conflict-free 16-byte reads, the chunk's weights (bulk-
//            async copy into shared memory, issued before phase A) as warp-wide broadcasts
//   phase C  threads 0..63, one column each: exp(-tau), Simpson scan over impact parameter
//            (modulation1, slantpath.c:350-436), first tau > toomuch -> last
// and the CTA leaves the chunk loop when every column has passed toomuch (tau.c:277-287), so the
// work follows the deepest column of the tile.  Summation order per (d, w) is i = 0..d, the same
// as the single-column form transit_column (tests/cpu_emu).
// The CTA is warp-specialised: warps 4-7 (PRODUCERS) only do phase A and run ahead through the
// chunks -- er[][] holds every layer, so they never wait for the consumers -- publishing each
// chunk through a shared-memory counter; warps 0-3 (CONSUMERS) do phases B and C behind their own
// named barrier.  The lookup's memory latency therefore overlaps the triangular product instead of
// alternating with it, and the SM holds 16 warps instead of 8.
constexpr int kTrW = 64, kTrThreads = 256, kTrCons = 128, kTrLoadBatch = 2, kTrMaxChunks = 16;
__device__ __forceinline__ void bar_consumers() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

template <int NMOL, int NCIA, bool KEEP>
__global__ void __launch_bounds__(kTrThreads, 2)
transit_tile_kernel(DevConfig c, const double *__restrict__ tabs, const double *__restrict__ wts,
                    const int *__restrict__ status, int *__restrict__ status_col,
                    double *__restrict__ spectra, double *__restrict__ tau_keep,
                    int *__restrict__ last_keep, int nmodels, int use_tma) {
  typedef TabLayout L;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar, bar_w;
  const int nl = c.nlayer, nf = c.lay.nf(), nd = c.lay.stride();
  unsigned long long *s_etab = reinterpret_cast<unsigned long long *>(smem_raw);
  double *s_tab = reinterpret_cast<double *>(s_etab + kExpTabSize);
  double *s_wt = s_tab + nd;                                   // [<= nl][kTrRow]
  double *s_er = s_wt + (size_t)nl * kTrRow;                   // [nl][kTrW]
  double *s_tau = s_er + (size_t)nl * kTrW;                    // [kTrChunk][kTrW]
  double *s_fd = s_tau + (size_t)kTrChunk * kTrW;              // [kTrChunk][kTrW] exp(-tau) b
  __shared__ __align__(8) uint64_t s_ready[kTrMaxChunks];      // mbarriers: the chunk's producer warps arrive
  __shared__ int s_stop, s_alive[2];                           // [chunk parity]
  const int m = blockIdx.x % nmodels;
  const int tile = blockIdx.x / nmodels;
  const bool producer = threadIdx.x >= kTrCons;
  const int t = producer ? threadIdx.x - kTrCons : threadIdx.x;   // index inside the role
  const int lane = t & 31, warp = t >> 5;
  const int wl = t & (kTrW - 1), dh = t >> 6;                  // lookup mapping: column, depth parity
  const int wcol = tile * kTrW + wl;
  const bool valid = wcol < c.nwave;
  const int w = valid ? wcol : c.nwave - 1;                    // columns past the end shadow the last one
  if (status[m] != 0) {                                        // rejected model: -1 fill
    if (!producer && t < kTrW && valid) spectra[(size_t)m * c.nwave + w] = -1.0;
    return;
  }
  if (threadIdx.x == 0) { mbar_init(&bar_w, 1); s_stop = 0; s_alive[0] = s_alive[1] = 0; }
  if (threadIdx.x < kTrMaxChunks) mbar_init(&s_ready[threadIdx.x], kTrCons / 32);
  fence_mbar_init();
  stage_table(s_tab, tabs + (size_t)m * nd, nd, &bar, use_tma != 0, s_etab);
  __syncthreads();
  const int nchunks = tr_nchunks(nl);
  const double wn = c.wn[w];

  if (producer) {
    // ---- phase A for every chunk: kTrChunk / 2 layers per thread, batches of independent loads
    const ColPtrs P = col_ptrs<NCIA>(c, w);
    const double wn4 = (wn * wn) * (wn * wn);
    for (int ch = 0; ch < nchunks; ch++) {
      if (*(volatile int *)&s_stop) break;                     // every column is past toomuch
      const int d0 = ch * kTrChunk;
#pragma unroll
      for (int j0 = 0; j0 < kTrChunk / 2; j0 += kTrLoadBatch) {
        CellData<NMOL, NCIA> x[kTrLoadBatch];
#pragma unroll
        for (int j = 0; j < kTrLoadBatch; j++) {
          const int d = d0 + dh + 2 * (j0 + j);
          if (d < nl) cell_load<NMOL, NCIA>(c, P, s_tab + (size_t)d * nf, x[j]);
        }
#pragma unroll
        for (int j = 0; j < kTrLoadBatch; j++) {
          const int d = d0 + dh + 2 * (j0 + j);
          if (d < nl)
            s_er[(size_t)d * kTrW + wl] = cell_combine<NMOL, NCIA>(c, P, s_tab + (size_t)d * nf, x[j], wn4, false);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_ready[ch]);
    }
    return;
  }

  // ---- consumers
  const double *wm = wts + (size_t)m * tr_stride(nl);
  double *tk = KEEP ? tau_keep + ((size_t)m * c.nwave + w) * nl : nullptr;
  // per-column state of phase C (threads 0..63)
  double S = 0.0, f1 = 0.0, f2 = 0.0, tau = 0.0, tau_prev = 0.0;
  int last = nl - 1;
  bool done = false;
  uint32_t wphase = 0;
  bool pending = false;                                        // a weight copy is in flight
  auto stage_weights = [&](int ch) {
    pending = true;
    const int rows = tr_rows(nl, ch);
    const double *wsrc = wm + tr_chunk_off(nl, ch);
    if (use_tma) {
      if (t == 0) {
        const uint32_t bytes = (uint32_t)rows * kTrRow * 8u;
        mbar_expect_tx(&bar_w, bytes);
        bulk_g2s(s_wt, wsrc, bytes, &bar_w);
      }
    } else {
      for (int i = t; i < rows * kTrRow; i += kTrCons) s_wt[i] = wsrc[i];
    }
  };
  stage_weights(0);
  for (int ch = 0; ch < nchunks; ch++) {
    const int d0 = ch * kTrChunk;
    const int dn = min(kTrChunk, nl - d0);
    // the chunk's extinction rows (and, by program order of the producers, all earlier ones)
    mbar_wait(&s_ready[ch], 0);
    if (use_tma) { mbar_wait(&bar_w, wphase); wphase ^= 1u; }
    else bar_consumers();
    pending = false;
    // ---- phase B: tau of depths d0 + 5 warp .. + 4 for columns 2 lane, 2 lane + 1
    {
      const int dg = d0 + kTrTD * warp;
      if (dg < nl) {
        const int kmax = min(dg + kTrTD - 1, nl - 1);
        double a0[kTrTD], a1[kTrTD];
#pragma unroll
        for (int j = 0; j < kTrTD; j++) { a0[j] = 0.0; a1[j] = 0.0; }
        const double *wr = s_wt + warp * kTrGroup;
        const double *ep = s_er + 2 * lane;
#pragma unroll 4
        for (int i = 0; i <= kmax; i++) {
          const D2 e = ld2(ep + (size_t)i * kTrW);
          const D2 w01 = ld2(wr + (size_t)i * kTrRow), w23 = ld2(wr + (size_t)i * kTrRow + 2);
          const double w4 = wr[(size_t)i * kTrRow + 4];
          a0[0] = fma(w01.x, e.x, a0[0]); a1[0] = fma(w01.x, e.y, a1[0]);
          a0[1] = fma(w01.y, e.x, a0[1]); a1[1] = fma(w01.y, e.y, a1[1]);
          a0[2] = fma(w23.x, e.x, a0[2]); a1[2] = fma(w23.x, e.y, a1[2]);
          a0[3] = fma(w23.y, e.x, a0[3]); a1[3] = fma(w23.y, e.y, a1[3]);
          a0[4] = fma(w4, e.x, a0[4]);    a1[4] = fma(w4, e.y, a1[4]);
        }
        // epilogue: the transmission integrand exp(-tau) b of every (depth, column) of the tile, all
        // threads, independent exponentials (phase C only scans)
#pragma unroll
        for (int j = 0; j < kTrTD; j++)
          if (dg + j < nl) {
            const double bd = s_tab[(size_t)(dg + j) * nf + L::RAD] * c.rfct;
            D2 v; v.x = a0[j]; v.y = a1[j];
            D2 f;
            f.x = fast_exp_neg(-v.x, s_etab) * bd;
            f.y = fast_exp_neg(-v.y, s_etab) * bd;
            *reinterpret_cast<D2 *>(s_tau + (size_t)(kTrTD * warp + j) * kTrW + 2 * lane) = v;
            *reinterpret_cast<D2 *>(s_fd + (size_t)(kTrTD * warp + j) * kTrW + 2 * lane) = f;
          }
      }
    }
    if (t == 0) s_alive[ch & 1] = 0;                           // last read two chunks ago
    bar_consumers();
    // the weight buffer is free: fetch the next chunk's while phase C runs
    if (ch + 1 < nchunks) stage_weights(ch + 1);
    // ---- phase C: one thread per column; branch-free so the loads and the panel products of the
    // chunk overlap (only the running sum S is a dependent chain, in the reference's order)
    if (t < kTrW && !done) {
      const double *tc = s_tau + t, *fc = s_fd + t;
      int jstop = kTrChunk;                                      // first depth of the chunk beyond toomuch
#pragma unroll
      for (int j = kTrChunk - 1; j >= 0; j--)
        if (j < dn && tc[(size_t)j * kTrW] > c.toomuch) jstop = j;
      const int jl = jstop < dn ? jstop : dn - 1;                // last depth processed in this chunk
      if (KEEP && valid)
        for (int j = 0; j <= jl; j++) tk[d0 + j] = tc[(size_t)j * kTrW];
#pragma unroll
      for (int j = 0; j < kTrChunk; j++) {
        const double fd = fc[(size_t)j * kTrW];
        if (j <= jl) {
          if (!(j & 1) && d0 + j >= 2) {                         // d0 is even: parity of d = parity of j
            const double *row = s_tab + (size_t)(d0 + j) * nf;
            S += row[L::SA] * fd + row[L::SB] * f1 + row[L::SC] * f2;
          }
          f2 = f1; f1 = fd;
        }
      }
      tau_prev = jl > 0 ? tc[(size_t)(jl - 1) * kTrW] : tau;     // tau still holds depth d0-1's
      tau = tc[(size_t)jl * kTrW];
      if (jstop < dn) { last = d0 + jstop; done = true; }
      if (!done) s_alive[ch & 1] = 1;
    }
    bar_consumers();
    if (!*(volatile int *)&s_alive[ch & 1]) { if (t == 0) s_stop = 1; break; }
  }
  // a bulk copy issued for a chunk that is never consumed must land before the CTA exits
  if (use_tma && pending) mbar_wait(&bar_w, wphase);
  if (t >= kTrW || !valid) return;
  if (KEEP) last_keep[(size_t)m * c.nwave + w] = last;
  if (c.modlevel == -1) {                                      // modulationm1 (slantpath.c:446-473)
    const int i0 = last > 0 ? last - 1 : 0;
    int st = 0;
    const double r = modulation_m1(tau_prev, tau, s_tab[(size_t)i0 * nf + L::RAD] * c.rfct,
                                   s_tab[(size_t)(i0 + 1) * nf + L::RAD] * c.rfct, c.toomuch,
                                   c.inv_srad2, &st);
    if (st) atomicOr(&status_col[m], st);
    spectra[(size_t)m * c.nwave + w] = r;
    return;
  }
  // modulation1 (slantpath.c:350-436): same tail as transit_column
  int n;
  if (last < nl - 1) {
    const int dd = last + 1;                                   // appended zero-integrand point
    const double *row = s_tab + (size_t)dd * nf;
    if (dd >= 2 && !(dd & 1)) S += row[L::SB] * f1 + row[L::SC] * f2;
    f2 = f1; f1 = 0.0;
    n = dd + 1;
  } else n = nl;
  double res;
  if (n < 3) { atomicOr(&status_col[m], REJ_FEWPTS); res = -1.0; }
  else {
    if (!(n & 1)) S += s_tab[(size_t)(n - 1) * nf + L::TR] * (f1 + f2);
    const double btop = s_tab[L::RAD] * c.rfct;
    res = btop * btop - 2.0 * S;
    if (c.transparent) {
      const double maxtau = tau > c.toomuch ? tau : c.toomuch;
      const double bl = s_tab[(size_t)(n - 1) * nf + L::RAD] * c.rfct;
      res -= fast_exp_neg(-maxtau, s_etab) * bl * bl;
    }
    res *= c.inv_srad2;
  }
  spectra[(size_t)m * c.nwave + w] = res;
}

// transit_mma_kernel: the same CTA shape and producer / consumer split, with the chord optical
// depth evaluated on the fp64 tensor cores.  tau(d, w) = sum_{i<=d} W[d][i] er[i][w] is, per model,
// a lower-triangular 100 x 100 matrix times the 100 x 64 extinction tile -- the one dense
// contraction of the forward model.  With DFMA the product is bound by the shared-memory pipe
// (every 10 multiply-adds of a lane need one 16-byte extinction read and 40 bytes of weight
// broadcasts: l1tex 82 %, fp64 29 %); mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4, 64 multiply-adds per
// clock per SM like DFMA -- tools/dmma_microbench.cu) takes its operands as warp-wide fragments,
// 1 shared-memory wavefront per 128 multiply-adds instead of 1 per 36.
//   chunk = 16 depths; consumer warp w owns columns 16 w .. 16 w + 15: 2 x 2 accumulator
//   fragments (depths x columns), K loop over the layers 0 .. d0 + 15 in steps of 4 (the upper
//   depth block stops 8 layers earlier: its weights beyond the diagonal are zero);
//   er[layer][64] is stored with its columns XOR-swizzled by 4 (layer & 3), so that the B-fragment
//   read (lane -> layer lane%4, column lane/4) is conflict-free within each half-warp at a row
//   stride of 64; the tau / exp(-tau) b tiles are swizzled by 8 on odd depths for the C-fragment
//   stores;
//   the chunk's weights arrive by one bulk-async copy (TMA) issued while the previous chunk's
//   scan runs (layout: column_math.cuh mm_rs / mm_chunk_off).
// The sum over layers runs in ascending order in groups of four; it differs from the DFMA kernel's
// (and the reference's) by rounding only.
constexpr int kMmThreads = 256, kMmCons = 128, kMmW = 64, kMmLoadBatch = 1, kMmMaxChunks = 20;
__device__ __forceinline__ void dmma884(double (&acc)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(acc[0]), "+d"(acc[1]) : "d"(a), "d"(b));
}

template <int NMOL, int NCIA, bool KEEP, bool SC>
__global__ void __launch_bounds__(kMmThreads, 2)
transit_mma_kernel(DevConfig c, const double *__restrict__ tabs, const double *__restrict__ wts,
                   const int *__restrict__ status, int *__restrict__ status_col,
                   double *__restrict__ spectra, double *__restrict__ tau_keep,
                   int *__restrict__ last_keep, int nmodels, int use_tma) {
  typedef TabLayout L;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar, bar_w;
  const int nl = c.nlayer, nf = c.lay.nf(), nd = c.lay.stride();
  const int nchunks = mm_nchunks(nl), nlp = nchunks * kMmChunk;
  unsigned long long *s_etab = reinterpret_cast<unsigned long long *>(smem_raw);
  double *s_tab = reinterpret_cast<double *>(s_etab + kExpTabSize);
  double *s_wt = s_tab + nd;                                   // [16][mm_rs(last chunk)]
  double *s_er = s_wt + (size_t)kMmChunk * mm_rs(nchunks - 1); // [nlp][64], swizzled
  double *s_tau = s_er + (size_t)nlp * kMmW;                   // [16][64]
  double *s_fd = s_tau + (size_t)kMmChunk * kMmW;              // [16][64] exp(-tau) b
  __shared__ __align__(8) uint64_t s_ready[kMmMaxChunks];      // mbarriers: the chunk's producer warps arrive
  __shared__ int s_stop, s_alive[2];
  const int m = blockIdx.x % nmodels;
  const int tile = blockIdx.x / nmodels;
  const bool producer = threadIdx.x >= kMmCons;
  const int t = producer ? threadIdx.x - kMmCons : threadIdx.x;
  const int lane = t & 31, warp = t >> 5;
  const int wl = t & (kMmW - 1);
  const int wcol = tile * kMmW + wl;
  const bool valid = wcol < c.nwave;
  const int w = valid ? wcol : c.nwave - 1;
  if (status[m] != 0) {
    if (!producer && t < kMmW && valid) spectra[(size_t)m * c.nwave + w] = -1.0;
    return;
  }
  if (threadIdx.x == 0) { mbar_init(&bar_w, 1); s_stop = 0; s_alive[0] = s_alive[1] = 0; }
  if (threadIdx.x < kMmMaxChunks) mbar_init(&s_ready[threadIdx.x], kMmCons / 32);
  fence_mbar_init();
  // rows past the last layer: zero extinction (their weights are zero as well)
  for (int i = nl * kMmW + threadIdx.x; i < nlp * kMmW; i += kMmThreads) s_er[i] = 0.0;
  stage_table(s_tab, tabs + (size_t)m * nd, nd, &bar, use_tma != 0, s_etab);
  __syncthreads();
  const double wn = c.wn[w];

  if (producer) {
    // Lookup: producer warp pw fills the depths d = pw (mod 4) of every chunk for all 64 columns of
    // the tile, two columns per lane (lane, lane + 32) addressed from one base pointer, so a depth's
    // table record is read by one warp only.  The CIA samples are kept across the depths of one
    // bracket row (as in eclipse_columns).  Columns past the end of the spectrum read the padding.
    // (Measured alternative: two tensor-core warps with 16 x 32 tiles and six producer warps, the
    // next depth's loads in flight while the current one is combined -- 12.3 ms against 8.3 ms: the
    // second register stage spills.  Without a second stage, the next depth's loads issued column by
    // column under the other column's arithmetic: 7.87 against 7.73 ms; an L1 prefetch of the next
    // depth's samples: 7.99 against 7.74; the consumer warps looking up half of the first chunk
    // instead of waiting for it: 7.76 / 7.70 against 7.73 / 7.80 at the W12 / demo shapes, i.e. nothing.)
    const int wa = tile * kMmW + lane;
    const ColPtrs P = col_ptrs<NCIA>(c, wa);
    constexpr bool kStatic = CellData<NMOL, NCIA>::kStatic;
    const size_t gstep = (size_t)32 * (kStatic ? CellData<NMOL, NCIA>::NG : c.gms) * 8, cstep = (size_t)32 * 32;
    double wn4[2];
#pragma unroll
    for (int k = 0; k < 2; k++) {
      const double v = c.wn[min(wa + 32 * k, c.nwave - 1)];
      wn4[k] = (v * v) * (v * v);
    }
    // x[0][k].q holds the CIA samples of the current bracket rows: a load with `fresh` false leaves
    // them in place (one stage only: kMmLoadBatch is 1)
    static_assert(kMmLoadBatch == 1, "the CIA samples live in the single load stage");
    CellData<NMOL, NCIA> x[kMmLoadBatch][2];
    CellOffs<NCIA> have;
    bool first = true;
    for (int ch = 0; ch < nchunks; ch++) {
      if (*(volatile int *)&s_stop) break;
      const int d0 = ch * kMmChunk;
#pragma unroll
      for (int j0 = 0; j0 < kMmChunk / 4; j0 += kMmLoadBatch) {
        bool fresh[kMmLoadBatch];
#pragma unroll
        for (int j = 0; j < kMmLoadBatch; j++) {
          const int d = d0 + 4 * (j0 + j) + warp;
          fresh[j] = false;
          if (d < nl) {
            const CellOffs<NCIA> o = cell_offsets<NMOL, NCIA>(s_tab + (size_t)d * nf);
            fresh[j] = first;
#pragma unroll
            for (int f = 0; f < (NCIA > 0 ? NCIA : 0); f++) fresh[j] = fresh[j] || o.cia[f] != have.cia[f];
#pragma unroll
            for (int k = 0; k < 2; k++) cell_load_at<NMOL, NCIA>(c, P, o, x[j][k], k * gstep, k * cstep, fresh[j]);
            have = o;
            first = false;
          }
        }
#pragma unroll
        for (int j = 0; j < kMmLoadBatch; j++) {
          const int d = d0 + 4 * (j0 + j) + warp;
          if (d < nl) {
            // both columns are combined before either is stored: with no shared-memory store in
            // between, the depth's table record is read once for the two of them
            double ev[2];
#pragma unroll
            for (int k = 0; k < 2; k++) {
              ev[k] = cell_combine<NMOL, NCIA, SC>(c, P, s_tab + (size_t)d * nf, x[j][k], wn4[k], false, k * gstep, k * cstep);
            }
#pragma unroll
            for (int k = 0; k < 2; k++) s_er[(size_t)d * kMmW + ((lane + 32 * k) ^ ((d & 3) << 2))] = ev[k];
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_ready[ch]);
    }
    return;
  }

  // ---- consumers
  const double *wm = wts + (size_t)m * mm_stride(nl);
  double *tk = KEEP ? tau_keep + ((size_t)m * c.nwave + w) * nl : nullptr;
  double S = 0.0, f1 = 0.0, f2 = 0.0, tau = 0.0, tau_prev = 0.0;
  int last = nl - 1;
  bool done = false;
  uint32_t wphase = 0;
  bool pending = false;
  auto stage_weights = [&](int ch) {
    pending = true;
    const int n = kMmChunk * mm_rs(ch);
    const double *wsrc = wm + mm_chunk_off(ch);
    if (use_tma) {
      if (t == 0) {
        mbar_expect_tx(&bar_w, (uint32_t)n * 8u);
        bulk_g2s(s_wt, wsrc, (uint32_t)n * 8u, &bar_w);
      }
    } else {
      for (int i = t; i < n; i += kMmCons) s_wt[i] = wsrc[i];
    }
  };
  stage_weights(0);
  const int g = lane >> 2, tg = lane & 3;
  for (int ch = 0; ch < nchunks; ch++) {
    const int d0 = ch * kMmChunk;
    const int dn = min(kMmChunk, nl - d0);
    mbar_wait(&s_ready[ch], 0);
    if (use_tma) { mbar_wait(&bar_w, wphase); wphase ^= 1u; }
    else bar_consumers();
    pending = false;
    // ---- phase B: tau[16 depths][16 columns of this warp] on the tensor cores
    {
      const int rs = mm_rs(ch);
      double acc[2][2][2];
#pragma unroll
      for (int a = 0; a < 2; a++)
#pragma unroll
        for (int b = 0; b < 2; b++) acc[a][b][0] = acc[a][b][1] = 0.0;
      const double *ap = s_wt + (size_t)g * rs + tg;           // A: row g (+8), layer k0 + tg
      const int sw = tg << 2;                                  // k0 is a multiple of 4: layer & 3 = tg
      const double *bp = s_er + (size_t)tg * kMmW;             // B: layer k0 + tg, column 16 warp + g (+8)
      const int cb0 = (16 * warp + g) ^ sw, cb1 = (16 * warp + g + 8) ^ sw;
      const int kend0 = d0 + 8, kend1 = d0 + kMmChunk;
      int k0 = 0;
#pragma unroll 2
      for (; k0 < kend0; k0 += 4) {
        const double b0 = bp[(size_t)k0 * kMmW + cb0], b1 = bp[(size_t)k0 * kMmW + cb1];
        const double a0 = ap[k0], a1 = ap[(size_t)8 * rs + k0];
        dmma884(acc[0][0], a0, b0); dmma884(acc[0][1], a0, b1);
        dmma884(acc[1][0], a1, b0); dmma884(acc[1][1], a1, b1);
      }
      for (; k0 < kend1; k0 += 4) {                            // lower depth block only
        const double b0 = bp[(size_t)k0 * kMmW + cb0], b1 = bp[(size_t)k0 * kMmW + cb1];
        const double a1 = ap[(size_t)8 * rs + k0];
        dmma884(acc[1][0], a1, b0); dmma884(acc[1][1], a1, b1);
      }
      // epilogue: C fragment = rows g (+8), columns 2 tg, 2 tg + 1 of each 8-column block
#pragma unroll
      for (int a = 0; a < 2; a++) {
        const int dl = 8 * a + g;
        if (d0 + dl < nl) {
          const double bd = s_tab[(size_t)(d0 + dl) * nf + L::RAD] * c.rfct;
#pragma unroll
          for (int b = 0; b < 2; b++) {
            const int col = 16 * warp + 8 * b + 2 * tg;
            D2 v; v.x = acc[a][b][0]; v.y = acc[a][b][1];
            D2 f;
            f.x = fast_exp_neg(-v.x, s_etab) * bd;
            f.y = fast_exp_neg(-v.y, s_etab) * bd;
            const int cs = col ^ ((dl & 1) << 3);
            *reinterpret_cast<D2 *>(s_tau + (size_t)dl * kMmW + cs) = v;
            *reinterpret_cast<D2 *>(s_fd + (size_t)dl * kMmW + cs) = f;
          }
        }
      }
    }
    if (t == 0) s_alive[ch & 1] = 0;
    bar_consumers();
    if (ch + 1 < nchunks) stage_weights(ch + 1);
    // ---- phase C: one thread per column (same scan as transit_tile_kernel)
    if (t < kMmW && !done) {
      const double *tc = s_tau, *fc = s_fd;
      auto at = [&](int j) { return (size_t)j * kMmW + (t ^ ((j & 1) << 3)); };
      int jstop = kMmChunk;
#pragma unroll
      for (int j = kMmChunk - 1; j >= 0; j--)
        if (j < dn && tc[at(j)] > c.toomuch) jstop = j;
      const int jl = jstop < dn ? jstop : dn - 1;
      if (KEEP && valid)
        for (int j = 0; j <= jl; j++) tk[d0 + j] = tc[at(j)];
#pragma unroll
      for (int j = 0; j < kMmChunk; j++) {
        const double fd = fc[at(j)];
        if (j <= jl) {
          if (!(j & 1) && d0 + j >= 2) {
            const double *row = s_tab + (size_t)(d0 + j) * nf;
            S += row[L::SA] * fd + row[L::SB] * f1 + row[L::SC] * f2;
          }
          f2 = f1; f1 = fd;
        }
      }
      tau_prev = jl > 0 ? tc[at(jl - 1)] : tau;
      tau = tc[at(jl)];
      if (jstop < dn) { last = d0 + jstop; done = true; }
      if (!done) s_alive[ch & 1] = 1;
    }
    bar_consumers();
    if (!*(volatile int *)&s_alive[ch & 1]) { if (t == 0) s_stop = 1; break; }
  }
  if (use_tma && pending) mbar_wait(&bar_w, wphase);
  if (t >= kMmW || !valid) return;
  if (KEEP) last_keep[(size_t)m * c.nwave + w] = last;
  if (c.modlevel == -1) {
    const int i0 = last > 0 ? last - 1 : 0;
    int st = 0;
    const double r = modulation_m1(tau_prev, tau, s_tab[(size_t)i0 * nf + L::RAD] * c.rfct,
                                   s_tab[(size_t)(i0 + 1) * nf + L::RAD] * c.rfct, c.toomuch,
                                   c.inv_srad2, &st);
    if (st) atomicOr(&status_col[m], st);
    spectra[(size_t)m * c.nwave + w] = r;
    return;
  }
  int n;
  if (last < nl - 1) {
    const int dd = last + 1;
    const double *row = s_tab + (size_t)dd * nf;
    if (dd >= 2 && !(dd & 1)) S += row[L::SB] * f1 + row[L::SC] * f2;
    f2 = f1; f1 = 0.0;
    n = dd + 1;
  } else n = nl;
  double res;
  if (n < 3) { atomicOr(&status_col[m], REJ_FEWPTS); res = -1.0; }
  else {
    if (!(n & 1)) S += s_tab[(size_t)(n - 1) * nf + L::TR] * (f1 + f2);
    const double btop = s_tab[L::RAD] * c.rfct;
    res = btop * btop - 2.0 * S;
    if (c.transparent) {
      const double maxtau = tau > c.toomuch ? tau : c.toomuch;
      const double bl = s_tab[(size_t)(n - 1) * nf + L::RAD] * c.rfct;
      res -= fast_exp_neg(-maxtau, s_etab) * bl * bl;
    }
    res *= c.inv_srad2;
  }
  spectra[(size_t)m * c.nwave + w] = res;
}

__global__ void merge_status_kernel(int *status, const int *status_col, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) status[i] |= status_col[i];
}

// ---------------------------------------------------------------------------------------
// K1 stand-alone lookup: ext[m][layer][w], layer index bottom -> top like the reference's e[r][w]
constexpr int kLookupBatch = 8;
template <int NMOL>
__global__ void __launch_bounds__(kColThreads)
extinction_kernel(DevConfig c, const double *__restrict__ tabs, double *__restrict__ ext,
                  int nmodels, int mol_only, int use_tma) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ __align__(8) uint64_t bar;
  double *s_tab = reinterpret_cast<double *>(smem_raw);
  const int m = blockIdx.x % nmodels;
  const int tile = blockIdx.x / nmodels;
  const int w = tile * kColThreads + threadIdx.x;
  const int nd = c.lay.stride();
  stage_table(s_tab, tabs + (size_t)m * nd, nd, &bar, use_tma != 0);
  if (w >= c.nwave) return;
  const double wn = c.wn[w];
  const double wn4 = (wn * wn) * (wn * wn);
  const int nl = c.nlayer;
  // blockIdx.y splits the layers so that small batches still fill the machine
  const int per = (nl + gridDim.y - 1) / gridDim.y;
  const int d0 = blockIdx.y * per, d1 = min(nl, d0 + per);
  double *out = ext + (size_t)m * nl * c.nwave + w;
  const ColPtrs P = col_ptrs<-1>(c, w);
  // batches of kLookupBatch depths: all global loads of a batch are issued before the first is
  // consumed (the kernel is a pure stream: what bounds it is the number of bytes in flight)
  const int nf = c.lay.nf();
  for (int d = d0; d < d1; d += kLookupBatch) {
    CellData<NMOL, -1> x[kLookupBatch];
#pragma unroll
    for (int j = 0; j < kLookupBatch; j++)
      if (d + j < d1) cell_load<NMOL, -1>(c, P, s_tab + (size_t)(d + j) * nf, x[j]);
#pragma unroll
    for (int j = 0; j < kLookupBatch; j++)
      if (d + j < d1)
        out[(size_t)(nl - 1 - d - j) * c.nwave] =
            cell_combine<NMOL, -1>(c, P, s_tab + (size_t)(d + j) * nf, x[j], wn4, mol_only);
  }
}

// Grid upload: one chunk of (layer, temperature) cells in file order [cell][mol][wave] ->
// device layout [cell][wave][gms] (molecule innermost, zero padding when gms > nmol).
__global__ void grid_relayout_kernel(const double *__restrict__ in, double *__restrict__ out,
                                     int ncells, int nmol, int gms, int nwave) {
  const size_t total = (size_t)ncells * nwave;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total;
       i += (size_t)gridDim.x * blockDim.x) {
    const size_t cell = i / nwave, w = i % nwave;
    const double *src = in + cell * (size_t)nmol * nwave + w;
    double *dst = out + i * gms;
    for (int m = 0; m < gms; m++) dst[m] = m < nmol ? src[(size_t)m * nwave] : 0.0;
  }
}

// ---------------------------------------------------------------------------------------
// K4 band integration: one CTA per (model, filter); trapezoid of (spectrum/star*rprs^2)*weight
// over the filter's contiguous sample range (wine.py:177-199, BARTfunc.py:386-396).
//
// Fused all-gather (SURVEY 8e): with a peer window the CTA also stores its band flux straight into
// every rank's window over NVLink (slot = generation parity, block = this rank), and the last CTA
// of the launch -- after a system-scope fence -- releases this rank's arrival flag on every peer.
// No NCCL call, no extra launch on the producer side; peer_wait_copy_kernel is the consumer.
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ void peer_announce(const PeerOut &po) {
  __threadfence_system();
  const unsigned long long g = *po.gen;
  for (int r = 0; r < po.world; r++) st_release_sys(po.flags[r] + po.rank, g + 1);
}

__global__ void __launch_bounds__(128)
band_integrate_kernel(const double *__restrict__ spectra, const double *__restrict__ wn,
                      const int *__restrict__ fstart, const int *__restrict__ fcount,
                      const int *__restrict__ foffset, const double *__restrict__ weight,
                      const double *__restrict__ star, double rprs2, const int *__restrict__ status,
                      double *__restrict__ bandflux, int nfilters, int nwave, PeerOut po) {
  const int m = blockIdx.x, f = blockIdx.y;
  // (the four scalars are fetched together: at MC3's population sizes this kernel is a chain of
  // memory round trips, so the loop below also issues the loads of kBandUnroll trapezoids before it
  // touches the first; a thread's terms are added in the same order as ever)
  const int stat = status ? status[m] : 0;
  const int s0 = fstart[f], n = fcount[f], off = foffset[f];
  const bool rejected = stat != 0;                       // CTA-uniform
  double acc = 0.0;
  if (!rejected) {
    const double *sp = spectra + (size_t)m * nwave + s0;
    const double *x = wn + s0;
    const double *wt = weight + off;
    const double *st = star ? star + off : nullptr;
    constexpr int kBandUnroll = 4;
    for (int k0 = threadIdx.x; k0 < n - 1; k0 += kBandUnroll * blockDim.x) {
      double y0[kBandUnroll], y1[kBandUnroll], w0[kBandUnroll], w1[kBandUnroll], x0[kBandUnroll],
          x1[kBandUnroll], d0[kBandUnroll], d1[kBandUnroll];
#pragma unroll
      for (int u = 0; u < kBandUnroll; u++) {
        const int k = k0 + u * blockDim.x;
        const int kk = k < n - 1 ? k : 0;                // a slot past the end re-reads sample 0, unused
        y0[u] = sp[kk]; y1[u] = sp[kk + 1];
        w0[u] = wt[kk]; w1[u] = wt[kk + 1];
        x0[u] = x[kk]; x1[u] = x[kk + 1];
        d0[u] = st ? st[kk] : 1.0; d1[u] = st ? st[kk + 1] : 1.0;
      }
#pragma unroll
      for (int u = 0; u < kBandUnroll; u++) {
        if (k0 + u * (int)blockDim.x >= n - 1) break;
        double a = y0[u], b = y1[u];
        if (st) { a = a / d0[u] * rprs2; b = b / d1[u] * rprs2; }
        acc += (x1[u] - x0[u]) * (b * w1[u] + a * w0[u]);
      }
    }
  }
  // fixed-shape reduction: deterministic for a given launch configuration
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
  __shared__ double s_part[4];
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  __shared__ int s_copier;
  const size_t idx = (size_t)m * nfilters + f;
  if (threadIdx.x == 0) {
    bandflux[idx] = rejected ? -1.0 : 0.5 * ((s_part[0] + s_part[1]) + (s_part[2] + s_part[3]));
    s_copier = 0;
    if (po.world > 0) {
      // models are handed to the peers in groups of kPeerGroup: the CTA that completes a group
      // ships it (so the system-scope fences are per group, not per band flux)
      __threadfence();
      const int grp = m / kPeerGroup;
      const int in_grp = (min((grp + 1) * kPeerGroup, (int)gridDim.x) - grp * kPeerGroup) * nfilters;
      if (atomicAdd(po.grpcnt + grp, 1u) == (unsigned)in_grp - 1) { s_copier = 1; __threadfence(); }
    }
  }
  __syncthreads();
  if (!s_copier) return;
  {
    const int grp = m / kPeerGroup;
    const size_t lo = (size_t)grp * kPeerGroup * nfilters;
    const size_t hi = (size_t)min((grp + 1) * kPeerGroup, (int)gridDim.x) * nfilters;
    const size_t slot = (size_t)(*po.gen & 1ull) * po.world * po.cap + (size_t)po.rank * po.cap;
    for (size_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
      const double v = __ldcg(bandflux + i);              // written by other CTAs: read at L2
      for (int r = 0; r < po.world; r++) po.win[r][slot + i] = v;
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
      po.grpcnt[grp] = 0;
      const unsigned int ngrp = (gridDim.x + kPeerGroup - 1) / kPeerGroup;
      if (atomicAdd(po.done, 1u) == ngrp - 1) {           // last group: everything is on its way
        *po.done = 0;
        peer_announce(po);
      }
    }
  }
}

__global__ void peer_signal_kernel(PeerOut po) { peer_announce(po); }

// Consumer: every CTA acquires all arrival flags (they are only polled, never written here), copies
// its slice of the generation's blocks, and the last CTA to finish advances the generation.
__global__ void __launch_bounds__(256)
peer_wait_copy_kernel(const double *__restrict__ win, unsigned long long *flags,
                      unsigned long long *gen, int world, long long cap, long long count,
                      double *__restrict__ out, int *err, unsigned int *finished,
                      unsigned long long timeout_ns) {
  __shared__ int s_bad;
  const unsigned long long g = *gen;            // advanced only after every CTA has passed this read
  if (threadIdx.x == 0) s_bad = 0;
  __syncthreads();
  if (threadIdx.x < world) {
    const unsigned long long t0 = global_ns();
    while (ld_acquire_sys(flags + threadIdx.x) < g + 1) {
      if (global_ns() - t0 > timeout_ns) { s_bad = 1; break; }            // a peer died or lags badly
      __nanosleep(200);
    }
  }
  __syncthreads();
  if (s_bad) { if (threadIdx.x == 0) *err = 1; }
  const double *src = win + (size_t)(g & 1ull) * world * cap;
  const long long total = (long long)world * count;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / count, k = i - r * count;
    out[i] = __ldcg(src + r * cap + k);                   // written by peers: bypass L1
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(finished, 1u) == gridDim.x - 1) { *finished = 0; __threadfence(); *gen = g + 1; }
  }
}

// L2 flush helper: stream-write a buffer larger than the L2
__global__ void fill_kernel(double *p, size_t n, double v) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    p[i] = v;
}

// ---------------------------------------------------------------------------------------
// launchers
static size_t table_smem(const DevConfig &c) {
  return ((size_t)c.lay.stride() + kExpTabSize) * sizeof(double);
}

void upload_exp_table(const DevConfig &c, cudaStream_t s) {
  unsigned long long h[(1 + kMaxAng) * kExpTabSize] = {};
  fill_ecl_exp_table(c, h);
  cudaMemcpyToSymbolAsync(g_exp_table, h, sizeof(h), 0, cudaMemcpyHostToDevice, s);
  cudaStreamSynchronize(s);
}

// Dynamic shared memory of the column kernels.  Every launch stages the model's whole table (one
// record per layer), so the shared memory of one block bounds the layer count a configuration can
// run: column_smem_fits() below holds these sizes against the device.
static size_t eclipse_smem(const DevConfig &c) {          // throughput, slot and scan kernels
  return ((size_t)c.lay.stride() + ecl_tab_entries(c.nang)) * sizeof(double);
}
static size_t transit_tile_smem(const DevConfig &c) {     // the DFMA tile kernel
  return table_smem(c) + ((size_t)c.nlayer * (kTrRow + kTrW) + (size_t)2 * kTrChunk * kTrW) * sizeof(double);
}

// Specialised instantiations for the shapes BART runs: f(nmol, ncia) with the grid-molecule and CIA
// counts as std::integral_constant, (1..4, 0..2) when both are in range, else the run-time-count
// build (0, -1).  dispatch_nmol is the molecule half: 1..4, else 0.
template <class F>
static void dispatch_nmol(int ngmol, F &&f) {
  switch (ngmol) {
    case 1: f(std::integral_constant<int, 1>()); break;
    case 2: f(std::integral_constant<int, 2>()); break;
    case 3: f(std::integral_constant<int, 3>()); break;
    case 4: f(std::integral_constant<int, 4>()); break;
    default: f(std::integral_constant<int, 0>());
  }
}
template <class F>
static void dispatch_counts(const DevConfig &c, F &&f) {
  dispatch_nmol(c.ngmol, [&](auto nmol) {
    const auto generic = [&] { f(std::integral_constant<int, 0>(), std::integral_constant<int, -1>()); };
    if constexpr (decltype(nmol)::value == 0) {
      generic();
    } else {
      switch (c.ncia) {
        case 0: f(nmol, std::integral_constant<int, 0>()); break;
        case 1: f(nmol, std::integral_constant<int, 1>()); break;
        case 2: f(nmol, std::integral_constant<int, 2>()); break;
        default: generic();
      }
    }
  });
}

void launch_grid_relayout(const double *in, double *out, int ncells, int nmol, int gms, int nwave,
                          cudaStream_t s) {
  grid_relayout_kernel<<<148 * 8, 256, 0, s>>>(in, out, ncells, nmol, gms, nwave);
}

void launch_atm_prep(const DevConfig &c, const Knobs &k, const double *profiles, int n_in,
                     double *tabs, int *status, const int *pre_status, int nmodels,
                     cudaStream_t s) {
  // staged through shared memory when it fits comfortably (W12: 41 KB), else the plain form
  size_t smem = atm_prep_smem_doubles(c) * sizeof(double);
  const int staged = smem <= 160 * 1024;
  if (!staged) smem = ((size_t)c.nspec + 3) * c.nlayer * sizeof(double);
  if (!allow_dyn_smem<atm_prep_kernel>(smem)) return;
  atm_prep_kernel<<<nmodels, kPrepThreads, smem, s>>>(c, k, profiles, n_in, tabs, status, pre_status, nmodels, staged);
}

// scan-kernel launch (specialised instantiations only; `if constexpr` keeps the run-time-count forms
// from instantiating it)
template <int NMOL, int NCIA, int NANG, int SQ, bool SC>
static void launch_eclipse_scan(const DevConfig &c, const double *tabs, const int *status, double *spectra,
                                int nmodels, int use_tma, size_t smem, cudaStream_t s) {
  if (!allow_dyn_smem<eclipse_scan_kernel<NMOL, NCIA, NANG, SQ, SC>>(smem)) return;
  // about one resident wave of warp tasks (4 columns each): 148 SMs x 6 CTAs x 4 warps
  constexpr int kWarps = kScanThreads / 32;
  const long long tasks = ((long long)(c.nwave + kScanCols - 1) / kScanCols) * nmodels;
  int tpw = (int)((tasks + 148LL * 6 * kWarps - 1) / (148LL * 6 * kWarps));
  tpw = tpw < 1 ? 1 : (tpw > 8 ? 8 : tpw);
  const int per = kWarps * tpw * kScanCols;
  const int tiles = (c.nwave + per - 1) / per;
  eclipse_scan_kernel<NMOL, NCIA, NANG, SQ, SC><<<(unsigned)((size_t)tiles * nmodels), kScanThreads, smem, s>>>(
      c, tabs, status, spectra, nmodels, use_tma, tpw);
}

// small: 0 = throughput kernel, 1 = slot kernel, 2 = scan kernel (where it exists, else the slot kernel)
template <int NMOL, int NCIA, int NANG, bool KEEP, int SQ = -1, bool SC = true>
static void launch_eclipse_t(const DevConfig &c, const double *tabs, const int *status,
                             double *spectra, double *tau_keep, int *last_keep, int nmodels,
                             int use_tma, int small, cudaStream_t s) {
  const size_t smem = eclipse_smem(c);
  if constexpr (!KEEP && CellData<NMOL, NCIA>::kStaticCia) {
    if (small == 2) {
      launch_eclipse_scan<NMOL, NCIA, NANG, SQ, SC>(c, tabs, status, spectra, nmodels, use_tma, smem, s);
      return;
    }
  }
  if (small && !KEEP) {
    if (!allow_dyn_smem<eclipse_slot_kernel<NMOL, NCIA, NANG, SQ, SC>>(smem)) return;
    const int nslots = (c.nwave + 31) / 32;
    eclipse_slot_kernel<NMOL, NCIA, NANG, SQ, SC><<<(unsigned)((size_t)nslots * nmodels), 32, smem, s>>>(
        c, tabs, status, spectra, nmodels, use_tma);
    return;
  }
  const int per = kEclThreads * kEclCols;
  const int tiles = (c.nwave + per - 1) / per;
  // Up to one resident wave of 8 CTAs per SM the kernel is latency-bound and the form that loads
  // one depth ahead is faster (W12, 24 models: 66 against 85 us); beyond, the in-step loads and
  // their 10 CTAs per SM are (4096 models: 3.77 against 4.12 ms).  Both give the same spectra to the bit.
  auto launch = [&](auto ahead) {                   // one instantiation per form
    constexpr auto kern = eclipse_column_kernel<NMOL, NCIA, NANG, KEEP, SQ, SC, decltype(ahead)::value>;
    if (!allow_dyn_smem<kern>(smem)) return;
    kern<<<(unsigned)((size_t)tiles * nmodels), kEclThreads, smem, s>>>(c, tabs, status, spectra, tau_keep,
                                                                       last_keep, nmodels, use_tma);
  };
  if constexpr (CellData<NMOL, NCIA>::kStatic) {
    if ((long long)tiles * nmodels <= 8LL * 148) {
      launch(std::true_type());
      return;
    }
  }
  launch(std::false_type());
}

// The specialised eclipse builds take the default 5-angle ray grid as a compile-time count as well
// (with or without scattering / cloud terms); any other grid takes the run-time angle count.
template <int NMOL, int NCIA, bool SC>
static void launch_eclipse_nang(const DevConfig &c, const double *tabs, const int *status,
                                double *spectra, int nmodels, int use_tma, int small, cudaStream_t s) {
  // the default ray grid (0 20 40 60 80 degrees): exp(-tau/cos 60) = exp(-tau/cos 0)^2
  if (c.nang == 5 && c.sq_src == 0 && c.sq_dst == 3)
    launch_eclipse_t<NMOL, NCIA, 5, false, 0x03, SC>(c, tabs, status, spectra, nullptr, nullptr, nmodels, use_tma, small, s);
  else launch_eclipse_t<NMOL, NCIA, 0, false, -1, SC>(c, tabs, status, spectra, nullptr, nullptr, nmodels, use_tma, small, s);
}

// Which eclipse kernel a batch of `nmodels` takes: 0 = throughput kernel (two columns per thread),
// 1 = slot kernel (one warp per 32 columns, bit-identical to 0), 2 = scan kernel (lanes <-> layers).
// $BART_ECL_SMALL = 0 / 1 / 2 forces one.
int eclipse_small_mode(const DevConfig &c, int nmodels) {
  const char *e = getenv("BART_ECL_SMALL");
  if (e && *e) return atoi(e);
  // the scan kernel's time grows with the column count from the first model on; the throughput
  // kernel needs ~8 CTAs per SM to hide its latencies and the slot kernel's fourfold CTA count
  // bridges the two (measured at the W12 shape: DESIGN.md section 4)
  if ((long long)c.nwave * nmodels <= kScanMaxColumns) return 2;
  // the slot kernel (one resident wave of one-warp CTAs, ~8 per SM by shared memory) is what is left
  // for the configurations the scan kernel is not instantiated for
  const long long nslots = (c.nwave + 31) / 32;
  return nslots * nmodels <= 8LL * 148 ? 1 : 0;
}

// Dynamic shared memory one block of `kern` can have on the current device: the opt-in limit less
// the kernel's static shared memory (0 when either cannot be read).
static size_t dyn_smem_max(const void *kern) {
  int dev = 0, optin = 0;
  cudaFuncAttributes a{};
  if (cudaGetDevice(&dev) != cudaSuccess ||
      cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess ||
      cudaFuncGetAttributes(&a, kern) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return (size_t)optin > a.sharedSizeBytes ? (size_t)optin - a.sharedSizeBytes : 0;
}

// The static shared memory of a kernel family does not depend on its template arguments (the
// eclipse kernels declare one mbarrier, the transit tile kernel its chunk barriers and flags); the
// least room over the generic and introspection builds stands for every build.  Read once: a
// process drives one device.
static size_t eclipse_dyn_max() {
  static const size_t v = std::min({dyn_smem_max((const void *)eclipse_column_kernel<0, -1, 0, true, -1, true, false>),
                                    dyn_smem_max((const void *)eclipse_column_kernel<0, -1, 0, false, -1, true, false>),
                                    dyn_smem_max((const void *)eclipse_slot_kernel<0, -1, 0, -1, true>)});
  return v;
}
static size_t transit_tile_dyn_max() {
  static const size_t v = std::min(dyn_smem_max((const void *)transit_tile_kernel<0, -1, true>),
                                   dyn_smem_max((const void *)transit_tile_kernel<0, -1, false>));
  return v;
}

bool column_smem_fits(const DevConfig &c) {
  if (c.eclipse) return eclipse_smem(c) <= eclipse_dyn_max();
  // transit: the DFMA tile kernel serves the introspection launches and every launch the tensor-core
  // kernel is not chosen for (transit_uses_mma: well inside the same limit), so it has to fit
  return tr_nchunks(c.nlayer) <= kTrMaxChunks && transit_tile_smem(c) <= transit_tile_dyn_max();
}

int column_layer_limit(const DevConfig &c) {
  DevConfig t = c;
  int best = 0;
  for (int nl = 1;; nl++) {
    t.nlayer = t.lay.nl = nl;
    if (!column_smem_fits(t)) return best;
    best = nl;
  }
}

bool launch_eclipse(const DevConfig &c, const double *tabs, const int *status, double *spectra,
                    double *tau_keep, int *last_keep, int nmodels, bool keep, bool sc, int use_tma,
                    cudaStream_t s) {
  if (!column_smem_fits(c)) return false;
  if (keep) {   // introspection path: run-time counts, stores tau[] and last[]
    launch_eclipse_t<0, -1, 0, true>(c, tabs, status, spectra, tau_keep, last_keep, nmodels, use_tma, 0, s);
    return true;
  }
  const int small = eclipse_small_mode(c, nmodels);
  if (c.planck_generic) {   // extreme Planck exponents: the kernel with the per-column clamp, degree 5
    launch_eclipse_t<0, -1, 0, false>(c, tabs, status, spectra, nullptr, nullptr, nmodels, use_tma, small, s);
    return true;
  }
  dispatch_counts(c, [&](auto nmol, auto ncia) {
    constexpr int NMOL = decltype(nmol)::value, NCIA = decltype(ncia)::value;
    if constexpr (NCIA < 0)   // the run-time-count build always has the scattering / cloud terms
      launch_eclipse_t<0, -1, 0, false>(c, tabs, status, spectra, nullptr, nullptr, nmodels, use_tma, small, s);
    else if (sc) launch_eclipse_nang<NMOL, NCIA, true>(c, tabs, status, spectra, nmodels, use_tma, small, s);
    else launch_eclipse_nang<NMOL, NCIA, false>(c, tabs, status, spectra, nmodels, use_tma, small, s);
  });
  return true;
}

void launch_merge_status(int *status, const int *status_col, int nmodels, cudaStream_t s) {
  merge_status_kernel<<<(nmodels + 255) / 256, 256, 0, s>>>(status, status_col, nmodels);
}

size_t transit_weights_stride(int nlayer) { return std::max(tr_stride(nlayer), mm_stride(nlayer)); }

static size_t transit_mma_smem(const DevConfig &c) {
  const int nch = mm_nchunks(c.nlayer);
  return table_smem(c) + ((size_t)kMmChunk * mm_rs(nch - 1) + (size_t)nch * kMmChunk * kMmW +
                          (size_t)2 * kMmChunk * kMmW) * sizeof(double);
}
// the tensor-core tile kernel serves every production launch it has the shared memory for (two CTAs
// per SM up to ~100 layers, one up to ~200); $BART_TRANSIT_MMA=0 forces the DFMA kernel
bool transit_uses_mma(const DevConfig &c, bool keep) {
  if (keep) return false;
  if (const char *e = getenv("BART_TRANSIT_MMA")) { if (*e && atoi(e) == 0) return false; }
  return mm_nchunks(c.nlayer) <= kMmMaxChunks && transit_mma_smem(c) <= 200 * 1024;
}

template <int NMOL, int NCIA, bool KEEP>
static void launch_transit_tile(const DevConfig &c, const double *tabs, const double *wts,
                                const int *status, int *status_col, double *spectra, double *tau_keep,
                                int *last_keep, int nmodels, int use_tma, cudaStream_t s) {
  const size_t smem = transit_tile_smem(c);
  if (!allow_dyn_smem<transit_tile_kernel<NMOL, NCIA, KEEP>>(smem)) return;
  const int tiles = (c.nwave + kTrW - 1) / kTrW;
  transit_tile_kernel<NMOL, NCIA, KEEP><<<(unsigned)((size_t)tiles * nmodels), kTrThreads, smem, s>>>(
      c, tabs, wts, status, status_col, spectra, tau_keep, last_keep, nmodels, use_tma);
}

template <int NMOL, int NCIA, bool SC>
static void launch_transit_mma(const DevConfig &c, const double *tabs, const double *wts,
                               const int *status, int *status_col, double *spectra, int nmodels,
                               int use_tma, cudaStream_t s) {
  const size_t smem = transit_mma_smem(c);
  if (!allow_dyn_smem<transit_mma_kernel<NMOL, NCIA, false, SC>>(smem)) return;
  const int tiles = (c.nwave + kMmW - 1) / kMmW;
  transit_mma_kernel<NMOL, NCIA, false, SC><<<(unsigned)((size_t)tiles * nmodels), kMmThreads, smem, s>>>(
      c, tabs, wts, status, status_col, spectra, nullptr, nullptr, nmodels, use_tma);
}

void launch_transit_weights(const DevConfig &c, const double *tabs, double *wts, int nmodels,
                            bool keep, int *status_col, cudaStream_t s) {
  transit_weights_kernel<<<nmodels, kTwThreads, (size_t)c.nlayer * sizeof(double), s>>>(
      c, tabs, wts, nmodels, transit_uses_mma(c, keep) ? 1 : 0, status_col);
}

bool launch_transit(const DevConfig &c, const double *tabs, const double *wts, const int *status,
                    int *status_col, double *spectra, double *tau_keep, int *last_keep,
                    int nmodels, bool keep, bool sc, int use_tma, cudaStream_t s) {
  if (!column_smem_fits(c)) return false;
  if (keep) {   // introspection path: run-time counts, stores tau[] and last[]
    launch_transit_tile<0, -1, true>(c, tabs, wts, status, status_col, spectra, tau_keep, last_keep, nmodels, use_tma, s);
    return true;
  }
  const bool mma = transit_uses_mma(c, false);
  dispatch_counts(c, [&](auto nmol, auto ncia) {
    constexpr int NMOL = decltype(nmol)::value, NCIA = decltype(ncia)::value;
    if (!mma)
      launch_transit_tile<NMOL, NCIA, false>(c, tabs, wts, status, status_col, spectra, nullptr, nullptr, nmodels, use_tma, s);
    else if (sc) launch_transit_mma<NMOL, NCIA, true>(c, tabs, wts, status, status_col, spectra, nmodels, use_tma, s);
    else launch_transit_mma<NMOL, NCIA, false>(c, tabs, wts, status, status_col, spectra, nmodels, use_tma, s);
  });
  return true;
}

void launch_extinction(const DevConfig &c, const double *tabs, double *ext, int nmodels,
                       int mol_only, int layer_splits, int use_tma, cudaStream_t s) {
  const size_t smem = (size_t)c.lay.stride() * sizeof(double);
  const int tiles = (c.nwave + kColThreads - 1) / kColThreads;
  dim3 grid((unsigned)((size_t)tiles * nmodels), (unsigned)layer_splits);
  dispatch_nmol(c.ngmol, [&](auto nmol) {
    constexpr auto kern = extinction_kernel<decltype(nmol)::value>;
    if (!allow_dyn_smem<kern>(smem)) return;
    kern<<<grid, kColThreads, smem, s>>>(c, tabs, ext, nmodels, mol_only, use_tma);
  });
}

void launch_band_integrate(const double *spectra, const double *wn, const int *fstart,
                           const int *fcount, const int *foffset, const double *weight,
                           const double *star, double rprs2, const int *status, double *bandflux,
                           int nfilters, int nwave, int nmodels, cudaStream_t s,
                           const PeerOut *peers) {
  PeerOut po;
  if (peers) po = *peers; else { memset(&po, 0, sizeof(po)); }
  dim3 grid((unsigned)nmodels, (unsigned)nfilters);
  band_integrate_kernel<<<grid, 128, 0, s>>>(spectra, wn, fstart, fcount, foffset, weight, star,
                                             rprs2, status, bandflux, nfilters, nwave, po);
}

void launch_peer_signal(const PeerOut &po, cudaStream_t s) { peer_signal_kernel<<<1, 1, 0, s>>>(po); }

void launch_peer_wait_copy(const double *win_local, unsigned long long *flags_local,
                           unsigned long long *gen, int world, long long cap, long long count,
                           double *out, int *err, unsigned int *finished,
                           unsigned long long timeout_ns, cudaStream_t s) {
  const long long total = (long long)world * count;
  const int grid = (int)std::max<long long>(1, std::min<long long>(64, total / 2048));
  peer_wait_copy_kernel<<<grid, 256, 0, s>>>(win_local, flags_local, gen, world, cap, count, out, err, finished,
                                             timeout_ns);
}

void launch_fill(double *p, size_t n, double v, cudaStream_t s) {
  fill_kernel<<<148 * 8, 256, 0, s>>>(p, n, v);
}

}  // namespace bart
