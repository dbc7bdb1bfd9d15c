// builder.hpp -- opacity-grid builder (stage d: --justOpacity), implemented in builder.cu
#pragma once
#include "host.hpp"
#include <cuda_runtime.h>
#include <memory>
#include <string>
#include <vector>

namespace bart {

struct BuilderState;
void builder_free(BuilderState *b);
struct BuilderFree { void operator()(BuilderState *b) const { builder_free(b); } };
// The builder of a configuration: created by the first call that needs it, freed with it.
using BuilderPtr = std::unique_ptr<BuilderState, BuilderFree>;

// Build the whole grid (all temperatures) and write the opacity file (opacity.c:406-421 layout).
void builder_run_and_write(BuilderPtr &b, const Options &o, const Atmosphere &a,
                           const Molecules &m, Tli &t, const std::vector<double> &wn,
                           cudaStream_t s, const std::string &path);
// Build temperatures [t_begin, t_end) only; host_out[layer][t - t_begin][mol][wave].
void builder_slice(BuilderPtr &b, const Options &o, const Atmosphere &a, const Molecules &m,
                   Tli &t, const std::vector<double> &wn, cudaStream_t s, int t_begin, int t_end,
                   double *host_out);
// Line-by-line forward mode (no opacity file; tau.c:163-175,253-264 -> computemolext(permol=0)):
// total molecular extinction of ncell (model, layer) cells, each at its own temperature
// cell_T[c] with mass densities d_cell_dens[c][nspec] (device), written to d_out + cell_out[c]
// (nwave doubles per cell, device).
void builder_lbl_cells(BuilderPtr &b, const Options &o, const Atmosphere &a, const Molecules &m,
                       Tli &t, const std::vector<double> &wn, cudaStream_t s, int ncell,
                       const double *cell_T, const double *d_cell_dens, const long long *cell_out,
                       double *d_out);
long long builder_stats(BuilderState *b, long long *nlines, long long *ngroups, long long *neval);
// milliseconds spent in a build phase so far: "voigt_table","line_index","grouping_host","kmax",
// "strength","widths","accumulate","d2h"
double builder_phase_ms(BuilderState *b, const char *name);
long long builder_line_bins(BuilderState *b, long long *iown_out, long long capacity);
int builder_profile(BuilderState *b, int idop, int ilor, float *out, long long capacity,
                    long long *halfsize);

}  // namespace bart
