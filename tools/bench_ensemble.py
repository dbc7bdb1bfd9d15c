#!/usr/bin/env python
"""Ensembles of retrievals in one device loop at the WASP-12b eclipse shape (the set-up of
tools/bench_latency.py: PT_line + 4 abundance factors, 9 parameters of which 7 free, 10 chains).
For every ensemble size R it reports, under CUDA-graph replay,
  demc / snooker us_per_generation     one generation of R x 10 models
  retrieval_generations_per_s          R / (generation time)
  models_per_s                         R x 10 / (generation time)
and the wall time of driver.run_demc_ensemble for a fixed number of generations against R
sequential driver.run_demc calls on the same data and streams.  --draws host,device adds, per walk,
  <walk>_host_streams_wall_s      run_<walk>_ensemble with streams drawn on the host from the rngs
                                  (host drawing included)
  <walk>_host_draw_s              that host drawing on its own (demc_draws / snooker_draws)
  <walk>_host_draw_share          the two above's ratio
  <walk>_seeded_wall_s            run_<walk>_ensemble(seeds=...): streams drawn on the device
  <walk>_draw_kernel_ms_per_call  the draw launches of one seeded call of --wall-gens generations
                                  (bart_kernel_stats, a profiled call of its own)
The card's name, power limit and max SM clock are read in the same run.
usage: bench_ensemble.py [--sizes 1,2,4,8,16,32,64] [--gens 600] [--wall-gens 200]
                         [--draws host,device] [--out file]"""
import argparse, json, os, subprocess, sys, tempfile, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bart_b200 import api, driver, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--sizes", default="1,2,4,8,16,32,64")
ap.add_argument("--chains", type=int, default=10)
ap.add_argument("--gens", type=int, default=600)
ap.add_argument("--wall-gens", type=int, default=200)
ap.add_argument("--draws", default="", help="host,device: time the drivers with each stream source")
ap.add_argument("--out", default=None)
a = ap.parse_args()
sizes = [int(x) for x in a.sizes.split(",")]
draw_modes = [m for m in a.draws.split(",") if m]
assert all(m in ("host", "device") for m in draw_modes), a.draws


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


RSUN, RJUP, MJUP, AU, G = 6.955e10, 7.1492e9, 1.8986e30, 1.4959787e13, 6.67384e-8
PTARGS = (1.57 * RSUN, 6300.0, 100.0, 0.0229 * AU, 100.0 * G * 1.41 * MJUP / (1.79 * RJUP) ** 2)
tmp = tempfile.mkdtemp(prefix="bart_ens_")
case = synth.make_case(tmp, shape="w12", solution="eclipse", seed=2026)
tr = api.Transit(case["cfg"])
wn = tr.get_waveno_arr()
hc_k = 6.6260755e-27 * 2.99792458e10 / 1.380658e-16
star = 2 * 6.6260755e-27 * 2.99792458e10 ** 2 * wn ** 3 / np.expm1(hc_k * wn / 6300.0) * np.pi
start, count, weight, st = api.filters_from_files(wn, case["filters"], wn, star)
tr.set_filters(start, count, weight, st, 0.117)
tr.converter_init(case["press_bar"], case["species"], case["abund"], ("H2O", "CO2", "CO", "CH4"), "line",
                  pt_args=PTARGS)
params = np.array([-0.5, -0.2, 1.0, 0.0, 1.1, 0.3, -0.2, 0.1, 0.2])
pmin = np.array([-5.0, -3.0, -2.0, 0.0, 0.55, -9.0, -9.0, -9.0, -9.0])
pmax = np.array([2.0, 2.0, 3.0, 1.0, 1.4, 3.0, 3.0, 3.0, 3.0])
stepsize = np.array([0.05, 0.05, 0.0, 0.0, 0.01, 0.3, 0.3, 0.3, 0.3])
free = stepsize > 0
nfree, nch = int(free.sum()), a.chains
truth, status = tr.bandflux_from_params(params[None, :])
assert status[0] == 0
Rmax = max(sizes)
data = np.array([truth[0] * (1 + 0.01 * np.random.RandomState(100 + r).normal(size=truth.shape[1]))
                 for r in range(Rmax)])
uncert = 0.02 * np.abs(data)
starts = []
for r in range(Rmax):
    p0 = np.repeat(params[None, :], nch, 0)
    p0[:, free] += np.random.RandomState(200 + r).normal(0, 0.01, (nch, nfree))
    starts.append(p0)
starts = np.array(starts)
ngen, warm = a.gens, 50
demc = [driver.demc_draws(np.random.RandomState(300 + r), nch, warm + ngen, stepsize[free]) for r in range(Rmax)]
hsize = nch + 1
snk = [driver.snooker_draws(np.random.RandomState(400 + r), nch, nfree, warm + ngen, hsize, 1, stepsize[free],
                            pmin[free], pmax[free]) for r in range(Rmax)]


rows = []
for R in sizes:
    row = {"nretr": R, "models_per_generation": R * nch}
    # DE-MC: warm-up call (graph capture, lazily configured launches), then one timed call
    tr.mcmc_init_ensemble(starts[:R], pmin, pmax, stepsize, data[:R], uncert[:R])
    tr.mcmc_run(*driver.stack_demc_draws(demc[:R], 0, warm))
    streams = driver.stack_demc_draws(demc[:R], warm, warm + ngen)
    t0 = time.perf_counter()
    tr.mcmc_run(*streams)
    us = 1e6 * (time.perf_counter() - t0) / ngen
    row["demc_us_per_generation"] = us
    row["demc_retrieval_generations_per_s"] = R / us * 1e6
    row["demc_models_per_s"] = R * nch / us * 1e6
    row["demc_accept_rate"] = float(tr.mcmc_get("numaccept").sum()) / (R * nch * (warm + ngen))
    # snooker
    tr.mcmc_init_ensemble(starts[:R], pmin, pmax, stepsize, data[:R], uncert[:R])
    tr.mcmc_snooker_init(np.stack([d["z0"] for d in snk[:R]]), 1)
    tr.mcmc_run_snooker(*driver.stack_snooker_draws(snk[:R], 0, warm))
    streams = driver.stack_snooker_draws(snk[:R], warm, warm + ngen)
    t0 = time.perf_counter()
    tr.mcmc_run_snooker(*streams)
    us = 1e6 * (time.perf_counter() - t0) / ngen
    row["snooker_us_per_generation"] = us
    row["snooker_retrieval_generations_per_s"] = R / us * 1e6
    row["snooker_models_per_s"] = R * nch / us * 1e6
    # whole-driver wall time: one ensemble run against R lone runs, same data and streams
    wg = a.wall_gens
    dw = [{k: (v[:wg] if k in ("support", "unif", "ugamma") else v[:, :wg]) for k, v in d.items()} for d in demc[:R]]
    t0 = time.perf_counter()
    ens = driver.run_demc_ensemble(tr, data[:R], uncert[:R], list(starts[:R]), pmin, pmax, stepsize, wg * nch,
                                   nch, draws=dw)
    row["run_demc_ensemble_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    lone = [driver.run_demc(tr, data[r], uncert[r], starts[r], pmin, pmax, stepsize, wg * nch, nch, draws=dw[r])
            for r in range(R)]
    row["sequential_run_demc_s"] = time.perf_counter() - t0
    row["wall_generations"] = wg
    row["wall_speedup"] = row["sequential_run_demc_s"] / row["run_demc_ensemble_s"]
    # the default kernel selection is batch-size dependent (scan kernel for small batches), so the
    # lone and ensemble chains agree to the scan kernel's ~1e-10, bit for bit when both take the
    # same kernel family (tests/test_gpu_retrieval_ensemble.py)
    row["ensemble_equals_lone_allparams"] = all(np.array_equal(e["allparams"], l["allparams"])
                                                for e, l in zip(ens, lone))
    for walk in ("demc", "snooker") if draw_modes else ():
        run = driver.run_demc_ensemble if walk == "demc" else driver.run_snooker_ensemble
        rngs = lambda: [np.random.RandomState(600 + r) for r in range(R)]
        args = (tr, data[:R], uncert[:R], list(starts[:R]), pmin, pmax, stepsize, wg * nch, nch)
        if "host" in draw_modes:
            t0 = time.perf_counter()
            for g in rngs():
                if walk == "demc":
                    driver.demc_draws(g, nch, wg, stepsize[free])
                else:
                    driver.snooker_draws(g, nch, nfree, wg, hsize, 1, stepsize[free], pmin[free], pmax[free])
            row[walk + "_host_draw_s"] = time.perf_counter() - t0
            t0 = time.perf_counter()
            run(*args, rngs=rngs())
            row[walk + "_host_streams_wall_s"] = time.perf_counter() - t0
            row[walk + "_host_draw_share"] = row[walk + "_host_draw_s"] / row[walk + "_host_streams_wall_s"]
        if "device" in draw_modes:
            keys = [(700 + r, 1) for r in range(R)]
            t0 = time.perf_counter()
            run(*args, rngs=rngs(), seeds=keys)
            row[walk + "_seeded_wall_s"] = time.perf_counter() - t0
            tr.mcmc_init_ensemble(starts[:R], pmin, pmax, stepsize, data[:R], uncert[:R])
            if walk == "snooker":
                tr.mcmc_snooker_init(np.stack([d["z0"] for d in snk[:R]]), 1)
            tr.mcmc_seed(np.array(keys, dtype=np.uint64))
            L = api.lib()
            L.bart_profile_enable(1)
            L.bart_profile_reset()
            tr.mcmc_run_seeded(wg)
            L.bart_profile_enable(0)
            st = api.kernel_stats().get("mcmc_draws", dict(launches=0, ms=float("nan")))
            row[walk + "_draw_kernel_ms_per_call"] = st["ms"] / max(1, st["launches"])
            L.bart_profile_reset()
    rows.append(row)
    print(json.dumps(row), flush=True)

base = rows[0]
out = {"workload": "WASP-12b eclipse shape, %d chains per retrieval, 9 parameters (7 free: PT_line "
                   "kappa gamma1 beta + 4 abundances), CUDA-graph replay, default kernel selection" % nch,
       "device": api.device_info() if hasattr(api, "device_info") else None,
       "nvidia_smi_name_power_limit_max_sm_clock": gpu_info(),
       "generations_timed": ngen,
       "draws": draw_modes,
       "rows": rows,
       "demc_speedup_vs_R1_per_retrieval_generation": {
           r["nretr"]: r["demc_retrieval_generations_per_s"] / base["demc_retrieval_generations_per_s"]
           for r in rows} if base["nretr"] == 1 else None}
tr.free_memory()
s = json.dumps(out, indent=1, default=str)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(s + "\n")
print(s)
