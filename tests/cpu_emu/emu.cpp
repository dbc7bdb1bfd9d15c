// tests/cpu_emu/emu.cpp -- TEST-ONLY host emulation of the CUDA kernels' thread loops.
//
// The arithmetic of the forward model lives in bart_b200/csrc/column_math.cuh as inline
// host+device functions; the CUDA kernels are thin wrappers that map (model, wavenumber) to
// threads.  This file maps the same functions over plain loops on the host so that the math
// can be compared with the oracle in the CPU-only container (pytest -m "not gpu").  It is NOT
// part of the product: libbart_b200.so contains no host execution path, nothing under
// bart_b200/ links or loads this file, and the GPU parity tests never use it.
#include "../../bart_b200/csrc/host.hpp"
#include "../../bart_b200/csrc/column_math.cuh"
#include <cstdarg>
#include <cstring>
#include <cstdlib>
#include <stdexcept>
#include <cmath>

namespace bart {
int g_verb = 0;
static char g_msg[2048];
void fail(const char *fmt, ...) {
  va_list ap; va_start(ap, fmt); vsnprintf(g_msg, sizeof(g_msg), fmt, ap); va_end(ap);
  throw std::runtime_error(g_msg);
}
void warn(int, const char *, ...) {}
}  // namespace bart

using namespace bart;

// the throughput kernel's thread shape (kernels.hpp kEclThreads, kEclCols): a thread carries two
// columns kEclThreads apart, and the grid and the CIA tables are padded by kEclPad samples
constexpr int kThreads = 64, kCols = 2, kPad = kThreads * kCols;

struct Emu {
  Options opt; Atmosphere atm; Molecules mol; Tli tli; OpacityGrid og;
  std::vector<CiaTable> cia;
  std::vector<double> wn, grid, PQ[kMaxCia];
  DevConfig c{};
  Knobs k{};
  bool lbl = false;
};
static Emu *E = nullptr;

extern "C" {

const char *emu_error() { return g_msg; }

int emu_init(const char *cfg) {
  try {
    delete E; E = new Emu();
    const char *argv[] = {"transit", "-c", cfg, nullptr};
    parse_options(3, (char **)argv, E->opt);
    Options &o = E->opt;
    double lo = o.wnlow > 0 ? o.wnlow * o.wnfct : 1.0 / (o.wlhigh * o.wlfct);
    double hi = o.wnhigh > 0 ? o.wnhigh * o.wnfct : 1.0 / (o.wllow * o.wlfct);
    E->wn = make_sampling(lo, hi, o.wndelt, 1);
    read_atmosphere(o.atm, E->atm);
    read_molecules(o.molfile, E->atm, E->mol);
    read_tli_header(o.linedb, E->tli);
    DevConfig &c = E->c;
    E->lbl = o.opacityfile.empty();
    if (E->lbl) {
      // line-by-line mode (transit.cu do_init): the "grid" is the caller's ext[layer][wave]
      E->og = OpacityGrid();
      E->og.nmol = 1; E->og.ntemp = 2; E->og.nlayer = E->atm.nlayer(); E->og.nwave = (long)E->wn.size();
      E->og.temp = {E->tli.tmin, E->tli.tmax};
      E->og.molid = {E->mol.id[0]};
    } else if (!read_opacity_header(o.opacityfile, E->og)) fail("no opacity file");
    OpacityGrid &g = E->og;
    size_t n = E->lbl ? 0 : (size_t)g.nlayer * g.ntemp * g.nmol * g.nwave;
    std::vector<double> filegrid(n);
    if (!E->lbl) {
    FILE *f = fopen(o.opacityfile.c_str(), "rb");
    fseek(f, g.data_offset, SEEK_SET);
    if (fread(filegrid.data(), 8, n, f) != n) fail("short grid");
    fclose(f);
    }
    // the device layout of the grid: [layer][temp][wave][gms] (device.cuh)
    c.gms = g.nmol == 1 ? 1 : (int)((g.nmol + 1) / 2 * 2);
    E->grid.assign((size_t)g.nlayer * g.ntemp * g.nwave * c.gms + (size_t)kPad * c.gms, 0.0);
    c.lbl = E->lbl ? 1 : 0;
    c.lbl_model0 = 0; c.lbl_dens = nullptr;
    for (size_t cell = 0; !E->lbl && cell < (size_t)(g.nlayer * g.ntemp); cell++)
      for (long m = 0; m < g.nmol; m++)
        for (long w = 0; w < g.nwave; w++)
          E->grid[(cell * g.nwave + w) * c.gms + m] = filegrid[(cell * g.nmol + m) * g.nwave + w];
    c.nlayer = E->atm.nlayer(); c.nspec = E->atm.nspec(); c.nwave = (int)E->wn.size();
    c.ntemp = (int)g.ntemp; c.ngmol = (int)g.nmol;
    c.eclipse = o.solution == "eclipse"; c.transparent = o.transparent; c.modlevel = o.modlevel;
    c.grid = E->grid.data(); c.gtemp = g.temp.data(); c.wn = E->wn.data();
    c.press = E->atm.press.data(); c.mass = E->mol.mass.data(); c.pol = E->mol.pol.data();
    for (int m = 0; m < c.ngmol; m++)
      for (int j = 0; j < c.nspec; j++) if (E->mol.id[j] == g.molid[m]) c.gmol_spec[m] = j;
    E->cia.resize(o.csfiles.size());
    c.ncia = (int)o.csfiles.size();
    for (int i = 0; i < c.ncia; i++) {
      read_cia(o.csfiles[i], E->cia[i]);
      std::vector<double> P, Q;
      fold_cia_table(E->cia[i], E->wn, P, Q);
      E->PQ[i] = pack_cia_quads(P, Q, (int)E->cia[i].temp.size(), (int)E->wn.size(), kPad);
      c.ciaPQ[i] = E->PQ[i].data(); c.ciaT[i] = E->cia[i].temp.data();
      c.cia_nt[i] = (int)E->cia[i].temp.size();
      c.cia_nspec[i] = (int)E->cia[i].species.size();
      for (size_t s = 0; s < E->cia[i].species.size(); s++)
        for (int j = 0; j < c.nspec; j++) if (E->atm.species[j] == E->cia[i].species[s]) c.cia_spec[i][s] = j;
    }
    c.pfct = E->atm.pfct; c.rfct = E->atm.rfct; c.gsurf = o.gsurf; c.p0 = o.refpress; c.toomuch = o.toomuch;
    c.ref_layer = ref_layer_of(c.press, c.nlayer, c.p0);
    std::vector<double> ang;
    char *dup = strdup(o.raygrid.c_str());
    for (char *t = strtok(dup, " \t"); t; t = strtok(nullptr, " \t")) ang.push_back(atof(t));
    free(dup);
    c.nang = (int)ang.size();
    std::vector<double> area(c.nang + 1);
    area[0] = 0.0; area[c.nang] = 90.0 * kDEG;
    for (int a = 1; a < c.nang; a++) area[a] = (ang[a - 1] + ang[a]) * kDEG / 2.0;
    for (int a = 0; a < c.nang; a++) {
      c.inv_mu[a] = 1.0 / cos(ang[a] * kDEG);
      c.wgt[a] = pow(sin(area[a + 1]), 2.0) - pow(sin(area[a]), 2.0);
    }
    fill_angle_consts(c);
    // Planck chaining and the choice of the generic Planck term, as transit_init sets them
    const int nw = c.nwave;
    c.planck_cols = 0;
    if (c.eclipse && nw > kThreads) {
      c.planck_cols = kThreads;
      c.planck_step = cH * cLS / cKB * kThreads * (E->wn[nw - 1] - E->wn[0]) / (nw - 1);
    }
    const double tmin = g.temp[0], tmax = g.temp[g.ntemp - 1], c2 = cH * cLS / cKB;
    c.planck_generic = !(tmin > 0) || c2 * E->wn[nw - 1] / tmin > 690.0 || c2 * E->wn[0] / tmax < 0.1;
    double srad = o.starrad * kSUNRADIUS;
    c.inv_srad2 = 1.0 / (srad * srad);
    c.lay.nl = c.nlayer; c.lay.ngmol = c.ngmol; c.lay.ncia = c.ncia;
    Knobs &k = E->k;
    k = Knobs();
    k.r0_all = o.refradius; k.cloud_flag_all = o.cloud_flag; k.cloudext_all = o.cloudext;
    k.cloudtop_all = o.cloudtop; k.cloudbot_all = o.cloudbot;
    k.scat_flag_all = o.scat_flag; k.scat_logext_all = o.scat_logext;
    return 0;
  } catch (std::exception &) { return -1; }
}

// line-by-line mode: the molecular extinction ext[layer][wave] of the next emu_run calls (what the
// builder kernels write for one model; one zero row of padding like transit.cu's buffer)
void emu_set_lbl_ext(const double *ext) {
  const size_t n = (size_t)E->c.nlayer * E->c.nwave;
  E->grid.assign(n + E->c.nwave, 0.0);
  memcpy(E->grid.data(), ext, n * 8);
  E->c.grid = E->grid.data();
}

int emu_nwave() { return E ? E->c.nwave : 0; }
int emu_nlayer() { return E ? E->c.nlayer : 0; }
void emu_wn(double *out) { for (int i = 0; i < E->c.nwave; i++) out[i] = E->wn[i]; }
void emu_set_radius(double r) { E->k.r0_all = r; }
void emu_set_cloudtop(double t) { E->k.cloud_flag_all = 1; E->k.cloudext_all = 100; E->k.cloudtop_all = t; E->k.cloudbot_all = t + 10; }
void emu_set_scattering(int f, double v) { E->k.scat_flag_all = f; E->k.scat_logext_all = v; }

} // extern "C"

// atm_prep of one model: the table records tab[depth][record] and the radii; returns the status
static int prep_model(const double *in, std::vector<double> &tab, std::vector<double> &rad) {
  DevConfig &c = E->c;
  const int nl = c.nlayer, ns = c.nspec;
  std::vector<double> rho((size_t)ns * nl), mu(nl), hc(nl);
  tab.assign(c.lay.stride(), 0.0);
  rad.assign(nl, 0.0);
  int status = 0;
  for (int l = 0; l < nl; l++) status |= prep_layer(c, in, l, rho.data() + l, nl, &mu[l]);
  KnobVals kv = knobs_for(E->k, 0);
  for (int l = 0; l + 1 < nl; l++) hc[l] = hydro_coef(c, in, mu.data(), l);
  hydrostatic_radii(c, kv.r0, in, mu.data(), hc.data(), rad.data());
  for (int d = 0; d < nl; d++) status |= prep_table_row(c, kv, d, in, rho.data(), nl, rad.data(), tab.data());
  return status;
}

// The eclipse throughput kernel's column loop (kernels.cu eclipse_column_kernel) over every tile of
// kThreads x kCols columns: the same eclipse_columns instantiation, one emulated thread at a time
template <int NMOL, int NCIA, int NANG, int SQ, bool PGEN, bool SC, bool AHEAD>
static void throughput_tiles(const DevConfig &c, const double *tab, const unsigned long long *etab,
                             double *spectrum) {
  for (int t0 = 0; t0 < c.nwave; t0 += kThreads * kCols)
    for (int x = 0; x < kThreads; x++) {
      const int w0 = t0 + x;
      bool valid[kCols];
      double *tk[kCols];
      int *lk[kCols];
      double flux[kCols];
      for (int k = 0; k < kCols; k++) { valid[k] = w0 + k * kThreads < c.nwave; tk[k] = nullptr; lk[k] = nullptr; }
      eclipse_columns<NMOL, NCIA, NANG, false, kCols, SQ, true, kThreads, PGEN, SC, AHEAD>(c, tab, etab, w0, valid,
                                                                                         tk, lk, flux);
      for (int k = 0; k < kCols; k++) if (valid[k]) spectrum[w0 + k * kThreads] = flux[k];
    }
}

extern "C" {

// One eclipse model through the build launch_eclipse (kernels.cu) selects for the configuration: the
// specialised (grid molecules, CIA files) pair with the default ray grid by squaring or a run-time
// angle count, with or without the scattering / cloud terms, and the one-depth-ahead (ahead != 0)
// or the in-step load order; the run-time-count build with the generic Planck term otherwise.
// build[0..1] receives the (NMOL, NCIA) template arguments that ran (0, -1: run-time counts); a
// rejected model runs no build.
int emu_run_build(const double *in, int ahead, double *spectrum, int *build) {
  DevConfig &c = E->c;
  const Knobs &k = E->k;
  if (!c.eclipse) return -1;                                   // eclipse configurations only
  std::vector<double> tab, rad;
  const int status = prep_model(in, tab, rad);
  if (status) { for (int w = 0; w < c.nwave; w++) spectrum[w] = -1; return status; }
  alignas(16) unsigned long long etab[(1 + kMaxAng) * kExpTabSize];
  fill_ecl_exp_table(c, etab);
  const bool sc = k.scat_flag_all != 0 || (k.cloud_flag_all == 1 && k.cloudext_all != 0.0);
  const bool sq = c.nang == 5 && c.sq_src == 0 && c.sq_dst == 3;
  const double *t = tab.data();
  build[0] = 0; build[1] = -1;
  auto pair = [&](auto nmol, auto ncia) {
    constexpr int N = decltype(nmol)::value, C = decltype(ncia)::value;
    build[0] = N; build[1] = C;
    auto run = [&](auto sqc, auto scc, auto aheadc) {
      constexpr bool S = decltype(sqc)::value;
      throughput_tiles<N, C, S ? 5 : 0, S ? 0x03 : -1, false, decltype(scc)::value, decltype(aheadc)::value>(
          c, t, etab, spectrum);
    };
    auto by_ahead = [&](auto sqc, auto scc) {
      if (ahead) run(sqc, scc, std::true_type()); else run(sqc, scc, std::false_type());
    };
    auto by_sc = [&](auto sqc) { if (sc) by_ahead(sqc, std::true_type()); else by_ahead(sqc, std::false_type()); };
    if (sq) by_sc(std::true_type()); else by_sc(std::false_type());
  };
  auto by_ncia = [&](auto nmol) {
    switch (c.ncia) {
      case 0: pair(nmol, std::integral_constant<int, 0>()); return true;
      case 1: pair(nmol, std::integral_constant<int, 1>()); return true;
      case 2: pair(nmol, std::integral_constant<int, 2>()); return true;
    }
    return false;
  };
  bool specialised = false;
  if (!c.planck_generic) switch (c.ngmol) {
    case 1: specialised = by_ncia(std::integral_constant<int, 1>()); break;
    case 2: specialised = by_ncia(std::integral_constant<int, 2>()); break;
    case 3: specialised = by_ncia(std::integral_constant<int, 3>()); break;
    case 4: specialised = by_ncia(std::integral_constant<int, 4>()); break;
  }
  // the run-time-count build has one (in-step) form and always the scattering / cloud terms
  if (!specialised) throughput_tiles<0, -1, 0, -1, true, true, false>(c, t, etab, spectrum);
  return 0;
}

// one model; tau[nwave][nlayer], last[nwave], radius[nlayer] optional
int emu_run(const double *in, double *spectrum, double *tau, int *last, double *radius,
            double *ext_total) {
  DevConfig &c = E->c;
  const int nl = c.nlayer, nw = c.nwave;
  std::vector<double> tab, rad;
  int status = prep_model(in, tab, rad);
  if (radius) for (int l = 0; l < nl; l++) radius[l] = rad[l];
  if (status) { for (int w = 0; w < nw; w++) spectrum[w] = -1; return status; }
  std::vector<double> tk(nl), wts((size_t)nl * (nl + 1) / 2), er(nl);
  alignas(16) unsigned long long etab[(1 + kMaxAng) * kExpTabSize];
  fill_ecl_exp_table(c, etab);
  if (!c.eclipse) for (int d = 0; d < nl; d++) transit_weight_row(c, tab.data(), d, &wts[(size_t)d * (d + 1) / 2]);
  for (int w = 0; w < nw; w++) {
    int lk = 0;
    std::fill(tk.begin(), tk.end(), 0.0);
    if (c.eclipse) {
      // exercise both the specialised and the run-time-count instantiations
      if (c.nang == 5 && c.ngmol == 1 && c.ncia == 1) spectrum[w] = eclipse_column<1, 1, 5, true>(c, tab.data(), etab, w, tk.data(), &lk);
      else if (c.nang == 5 && c.ngmol == 4 && c.ncia == 1) spectrum[w] = eclipse_column<4, 1, 5, true>(c, tab.data(), etab, w, tk.data(), &lk);
      else spectrum[w] = eclipse_column<0, -1, 0, true>(c, tab.data(), etab, w, tk.data(), &lk);
    } else {
      spectrum[w] = transit_column<0, -1, true>(c, tab.data(), etab, wts.data(), w, er.data(), 1, tk.data(), &lk, &status);
    }
    if (tau) memcpy(tau + (size_t)w * nl, tk.data(), nl * 8);
    if (last) last[w] = lk;
    if (ext_total) {
      const double wn = c.wn[w], wn4 = (wn * wn) * (wn * wn);
      const ColPtrs P = col_ptrs<-1>(c, w);
      for (int d = 0; d < nl; d++)
        ext_total[(size_t)(nl - 1 - d) * nw + w] = cell_extinction<0, -1>(c, P, tab.data() + (size_t)d * c.lay.nf(), wn4, true);
    }
  }
  return status;
}

// host readers of the product (readers.cpp): the memory-mapped TLI line selection.  Returns the
// number of selected lines and copies up to `cap` of them.
long long emu_read_tli(const char *path, double wnlow, double wnhigh, long long cap, double *wl,
                       double *elow, double *gf, short *isoid) {
  try {
    Tli t;
    read_tli_header(path, t);
    read_tli_lines(path, t, wnlow, wnhigh);
    const long long n = (long long)t.wl.size();
    for (long long i = 0; i < n && i < cap; i++) { wl[i] = t.wl[i]; elow[i] = t.elow[i]; gf[i] = t.gf[i]; isoid[i] = t.isoid[i]; }
    return n;
  } catch (std::exception &) { return -1; }
}

// Chord optical depths through the DEVICE code's weight construction (column_math.cuh
// transit_weight_row_acc, what transit_weights_kernel runs per depth): radii by depth (top -> bottom),
// extinction by depth; tau[d] = sum_{i<=d} W[d][i] ex[i] / rfct'.  For the analytic known-answer
// tests of the reference's own test design (transit/test/test_slantpath.c:177-198).
void emu_chord_tau(int nl, const double *radius_by_depth, const double *ex_by_depth, double *tau) {
  DevConfig c{};
  c.nlayer = nl; c.rfct = 1.0;
  c.lay.nl = nl; c.lay.ngmol = 1; c.lay.ncia = 0;
  const int nf = c.lay.nf();
  std::vector<double> tab((size_t)nf * nl, 0.0), wt(nl);
  for (int d = 0; d < nl; d++) tab[(size_t)d * nf + TabLayout::RAD] = radius_by_depth[d];
  for (int d = 0; d < nl; d++) {
    transit_weight_row(c, tab.data(), d, wt.data());
    double t = 0.0;
    for (int i = 0; i <= d; i++) t += wt[i] * ex_by_depth[i];
    tau[d] = t;
  }
}

// A chord-weight row assembled from `nparts` shares of its panels (what transit_weights_kernel does
// with kTwParts threads per depth) against the whole row: number of elements that differ in any bit,
// over all depths.
int emu_chord_parts_mismatch(int nl, const double *radius_by_depth, int nparts) {
  DevConfig c{};
  c.nlayer = nl; c.rfct = 1e5;
  int bad = 0;
  std::vector<double> whole(nl), split(nl);
  for (int d = 0; d < nl; d++) {
    auto rad = [radius_by_depth](int i) { return radius_by_depth[i]; };
    std::fill(whole.begin(), whole.end(), -1.0);
    std::fill(split.begin(), split.end(), -1.0);
    double *w = whole.data(), *sp = split.data();
    transit_weight_row_parts(c, rad, d, [w](int i) -> double & { return w[i]; }, 0, 1);
    for (int k = 0; k < nparts; k++)
      transit_weight_row_parts(c, rad, d, [sp](int i) -> double & { return sp[i]; }, k, nparts);
    for (int i = 0; i < nl; i++) bad += memcmp(&whole[i], &split[i], 8) != 0;
    for (int i = 0; i <= d; i++) bad += whole[i] == -1.0;       // every element of the row is written
  }
  return bad;
}

double emu_fast_exp(double x) { unsigned long long t[kExpTabSize]; fill_exp_table(t); return fast_exp(x, t); }

}  // extern "C"
