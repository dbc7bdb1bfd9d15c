// kernels.hpp -- host-callable launchers of kernels.cu / builder.cu
#pragma once
#include "device.cuh"
#include <cuda_runtime.h>
#include <cstddef>

namespace bart {

constexpr int kColThreads = 128;      // wavenumbers per CTA, lookup kernel
constexpr int kEclThreads = 64;       // eclipse kernel: 64 threads x kEclCols columns = 128 wavenumbers per CTA
constexpr int kEclCols = 2;
// the eclipse kernel addresses a thread's columns from one base pointer and does not clamp the
// columns past the end of the spectrum: the grid, the CIA tables and the line-by-line extinction
// buffer carry this many samples of padding behind their last plane
constexpr int kEclPad = kEclThreads * kEclCols;

void launch_atm_prep(const DevConfig &c, const Knobs &k, const double *profiles, int n_in,
                     double *tabs, int *status, const int *pre_status, int nmodels,
                     cudaStream_t s);
// Whether the column kernels' shared memory (the model's table is staged whole) fits one block of
// the current device for configuration `c`; the largest layer count that does, the other counts of
// `c` unchanged.  launch_eclipse / launch_transit launch nothing and return false when it does not.
bool column_smem_fits(const DevConfig &c);
int column_layer_limit(const DevConfig &c);
// sc: some record of the launch may carry a scattering or cloud term (false: skipped altogether)
bool launch_eclipse(const DevConfig &c, const double *tabs, const int *status, double *spectra,
                    double *tau_keep, int *last_keep, int nmodels, bool keep, bool sc, int use_tma,
                    cudaStream_t s);
// chord weights of one model in the tiled layout (doubles per model), K2t, and the tile kernel
size_t transit_weights_stride(int nlayer);
// keep: the launch that follows is the introspection one (it takes the DFMA kernel's layout)
// status_col (or nullptr): the per-model column-status words of the launch that follows, cleared here
void launch_transit_weights(const DevConfig &c, const double *tabs, double *wts, int nmodels,
                            bool keep, int *status_col, cudaStream_t s);
bool launch_transit(const DevConfig &c, const double *tabs, const double *wts, const int *status,
                    int *status_col, double *spectra, double *tau_keep, int *last_keep,
                    int nmodels, bool keep, bool sc, int use_tma, cudaStream_t s);
void launch_merge_status(int *status, const int *status_col, int nmodels, cudaStream_t s);
// mol_only: 0 = total extinction, 1 = molecular lines only, 2 = CIA only
void launch_extinction(const DevConfig &c, const double *tabs, double *ext, int nmodels,
                       int mol_only, int layer_splits, int use_tma, cudaStream_t s);
// Peer window of the fused band-integration + all-gather (one process per GPU, windows mapped
// through CUDA IPC over NVLink/NVSwitch).  win[r] / flags[r] are rank r's window and arrival
// flags as seen from this process; a window holds 2 slots x world x cap doubles.
constexpr int kMaxPeers = 8;
constexpr int kPeerGroup = 64;        // models shipped to the peers per copier CTA
struct PeerOut {
  double *win[kMaxPeers];
  unsigned long long *flags[kMaxPeers];
  int world, rank;                    // world == 0: no peers (plain band integration)
  long long cap;                      // doubles per rank per slot
  const unsigned long long *gen;      // generation counter (device; advanced by the wait kernel)
  unsigned int *done;                 // completed groups of the launch
  unsigned int *grpcnt;               // [groups] completed CTAs per group of kPeerGroup models
};
// waits until every rank's block of generation *gen has arrived in the local window, copies
// world x count doubles to `out` ([rank][count]) and advances *gen; *err is set after timeout_ns
// without a peer's arrival flag (the copy still proceeds: the caller must check *err)
void launch_peer_wait_copy(const double *win_local, unsigned long long *flags_local,
                           unsigned long long *gen, int world, long long cap, long long count,
                           double *out, int *err, unsigned int *finished,
                           unsigned long long timeout_ns, cudaStream_t s);
// a rank with no model in this generation still has to announce itself
void launch_peer_signal(const PeerOut &po, cudaStream_t s);
void launch_band_integrate(const double *spectra, const double *wn, const int *fstart,
                           const int *fcount, const int *foffset, const double *weight,
                           const double *star, double rprs2, const int *status, double *bandflux,
                           int nfilters, int nwave, int nmodels, cudaStream_t s,
                           const PeerOut *peers = nullptr);
void launch_fill(double *p, size_t n, double v, cudaStream_t s);
void upload_exp_table(const DevConfig &c, cudaStream_t s);   // after fill_angle_consts
// [cell][mol][wave] (file order) -> [cell][wave][gms] (device order), ncells (layer, T) cells
void launch_grid_relayout(const double *in, double *out, int ncells, int nmol, int gms, int nwave,
                          cudaStream_t s);

}  // namespace bart
