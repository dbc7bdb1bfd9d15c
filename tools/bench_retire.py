#!/usr/bin/env python
"""Stopping retrievals of an ensemble early (bart_mcmc_retain, driver grexit="each") at the
WASP-12b eclipse shape of tools/bench_ensemble.py (PT_line + 4 abundance factors, 9 parameters of
which 7 free, 10 chains per retrieval), seeded snooker walk.  Reports
  retain[]        kernel time of one bart_mcmc_retain (mcmc_retain launch, CUDA events) from
                  64 retrievals to 32 and to 8 with histories of ~1e3 and ~1e4 rows; its HBM
                  traffic (the kept state read and written, unfilled history rows read once) and
                  that over the kernel time, against the 7.7 TB/s data-sheet HBM bandwidth
  after_retain    us per generation of a loop retained from 64 to 16 retrievals against a fresh
                  16-retrieval loop, alternated `--reps` times in this process
  end_to_end      wall time of run_snooker_ensemble(R = 64, seeds, grtest=True) with and without
                  grexit="each", each retrieval's exit iteration and the retrieval-generations run;
                  three retrievals in four have flat likelihoods and converge at
                  different checkpoints, the fourth does not converge; alternated `--reps` times
The card's name, power limit and max SM clock are read in the same run.
usage: bench_retire.py [--chains 10] [--reps 5] [--gens 300] [--chainsize 8000] [--out file]"""
import argparse, json, os, subprocess, sys, tempfile, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bart_b200 import api, driver, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--chains", type=int, default=10)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--gens", type=int, default=300)
ap.add_argument("--chainsize", type=int, default=8000)
ap.add_argument("--out", default=None)
a = ap.parse_args()

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip().splitlines()
gpu = q[0] if q else "unknown"

RSUN, RJUP, MJUP, AU, G = 6.955e10, 7.1492e9, 1.8986e30, 1.4959787e13, 6.67384e-8
PTARGS = (1.57 * RSUN, 6300.0, 100.0, 0.0229 * AU, 100.0 * G * 1.41 * MJUP / (1.79 * RJUP) ** 2)
tmp = tempfile.mkdtemp(prefix="bart_retire_")
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
nfree, nch, npars, R = int(free.sum()), a.chains, len(params), 64
truth, status = tr.bandflux_from_params(params[None, :])
assert status[0] == 0
ndata = truth.shape[1]
data = np.array([truth[0] * (1 + 0.01 * np.random.RandomState(100 + r).normal(size=ndata)) for r in range(R)])
uncert = 0.02 * np.abs(data)
starts = []
for r in range(R):
    p0 = np.repeat(params[None, :], nch, 0)
    p0[:, free] += np.random.RandomState(200 + r).normal(0, 0.01, (nch, nfree))
    starts.append(p0)
starts = np.array(starts)
hsize = nch + 1
z0 = np.stack([driver.snooker_z0(np.random.RandomState(400 + r), nch, hsize, pmin[free], pmax[free])
               for r in range(R)])
keys = np.array([(700 + r, 1) for r in range(R)], dtype=np.uint64)
L = api.lib()


def loop(idx, gens):
    """seeded snooker loop of retrievals idx after `gens` generations (one call)"""
    tr.mcmc_init_ensemble(starts[idx], pmin, pmax, stepsize, data[idx], uncert[idx])
    tr.mcmc_seed(keys[idx])
    tr.mcmc_snooker_init(z0[idx], 1)
    if gens:
        tr.mcmc_run_seeded(gens)


def zcap(rows_needed):
    """history rows allocated (snooker_reserve_rows: the rows asked for + half + 16)"""
    cap = hsize + 64
    cap += cap // 2 + 16
    if rows_needed > cap:
        cap = rows_needed + rows_needed // 2 + 16
    return cap


def retain_cost(rows, nkeep):
    gens = rows - hsize
    out = []
    for rep in range(2):
        loop(list(range(R)), gens)
        L.bart_profile_enable(1)
        L.bart_profile_reset()
        tr.mcmc_retain(list(range(0, R, R // nkeep)))
        L.bart_profile_enable(0)
        st = api.kernel_stats()["mcmc_retain"]
        out.append(st["ms"] / st["launches"])
        L.bart_profile_reset()
    cap = zcap(hsize + gens + 1)
    filled = hsize + gens
    # HBM traffic of the gather for the kept retrievals.  History (Z, Zchisq): the filled rows and
    # the one template row that every unfilled row is copied from (its later reads hit L2) are read,
    # every allocated row is written.  The rest is read and written once: doubles data, uncert,
    # bestmodel, bestp, bestchisq, zbest, key; per chain params, nextp, currchisq, nextchisq, c2,
    # numaccept, curmodel; ints iter, zsize; per chain outbounds, outflag, noproj, slot.
    zrow = 8 * nch * (npars + 1)
    rest = 8 * (4 * ndata + 2 * npars + 4 + nch * (2 * npars + 4 + ndata)) + 4 * (2 + nch * (nfree + 3))
    moved = nkeep * ((filled + 1) * zrow + cap * zrow + 2 * rest)
    ms = min(out)
    return {"rows": filled, "rows_allocated": cap, "from": R, "to": nkeep, "kernel_ms": out,
            "bytes_moved": moved, "achieved_TB_per_s": moved / (ms * 1e-3) / 1e12,
            "share_of_7.7_TB_per_s": moved / (ms * 1e-3) / 7.7e12}


res = {"workload": "WASP-12b eclipse shape, %d chains per retrieval, 9 parameters (7 free), seeded snooker, "
                   "thinning 1, CUDA-graph replay, default kernel selection" % nch,
       "nvidia_smi_name_power_limit_max_sm_clock": gpu, "retain": []}
for rows in (1000, 10000):
    for nkeep in (32, 8):
        res["retain"].append(retain_cost(rows, nkeep))
        print(json.dumps(res["retain"][-1]), flush=True)

# no cost left behind: a loop retained 64 -> 16 against a fresh 16, alternated
warm, ng = 60, a.gens
kept = list(range(0, R, 4))
times = {"retained_64_to_16": [], "fresh_16": []}
for rep in range(a.reps):
    for name in times:
        if name == "fresh_16":
            loop(kept, warm)
        else:
            loop(list(range(R)), warm)
            tr.mcmc_retain(list(range(0, R, 4)))
        tr.mcmc_run_seeded(20)                                     # graph capture at this size
        t0 = time.perf_counter()
        tr.mcmc_run_seeded(ng)
        times[name].append(1e6 * (time.perf_counter() - t0) / ng)
res["after_retain_us_per_generation"] = {k: dict(runs=v, median=float(np.median(v)), min=min(v), max=max(v))
                                         for k, v in times.items()}
print(json.dumps(res["after_retain_us_per_generation"]), flush=True)

# end to end: grexit="each" against grtest only, same keys.  Three retrievals in four have a flat
# likelihood (uncertainties scaled by 10^8 ... 10^4) and chains started uniformly in the free
# parameters' bounds, so DE-MC's jumps mix them within a few checkpoints; the fourth keeps its
# uncertainties and starts 3 step sizes around the truth, and does not converge in the run.
flat = np.arange(R) % 4 != 3
mult = np.where(flat, 10.0 ** np.linspace(8, 4, R), 1.0)
u2 = uncert * mult[:, None]
cs = a.chainsize
e2e_starts = []
for r in range(R):
    g = np.random.RandomState(300 + r)
    p0 = np.repeat(params[None, :], nch, 0)
    if flat[r]:
        p0[:, free] = g.uniform(pmin[free], pmax[free], (nch, nfree))
    else:
        p0[:, free] += g.normal(0, 3.0, (nch, nfree)) * stepsize[free]
    e2e_starts.append(np.clip(p0, pmin, pmax))
run = lambda **kw: driver.run_snooker_ensemble(tr, data, u2, e2e_starts, pmin, pmax, stepsize, cs * nch, nch,
                                                hsize=hsize, rngs=[np.random.RandomState(400 + r) for r in range(R)],
                                                seeds=[(800 + r, 3) for r in range(R)], grtest=True, **kw)
# host time of the state fetches and retains grexit="each" adds at the checkpoints where retrievals stop
host = {"state_fetch_s": 0.0, "retain_s": 0.0}
get, retain = tr.mcmc_get, tr.mcmc_retain


def timed(f, key, skip=()):
    def g(*args):
        t0 = time.perf_counter()
        v = f(*args)
        if args[0] not in skip:
            host[key] += time.perf_counter() - t0
        return v
    return g


tr.mcmc_get = timed(get, "state_fetch_s", skip=("allparams", "allmodel"))
tr.mcmc_retain = lambda keep: timed(retain, "retain_s")(keep)
walls = {"grtest_only": [], "grexit_each": []}
e2e = {}
for rep in range(a.reps):
    for name, kw in (("grtest_only", {}), ("grexit_each", dict(grexit="each"))):
        host.update(state_fetch_s=0.0, retain_s=0.0)
        t0 = time.perf_counter()
        outs = run(**kw)
        walls[name].append(time.perf_counter() - t0)
        e2e[name + "_host_state_fetch_s"] = host["state_fetch_s"]
        if name == "grexit_each":
            e2e["grexit_each_host_retain_s"] = host["retain_s"]
            lengths = [int(o["allparams"].shape[-1]) for o in outs]
            e2e["exit_iteration"] = lengths
            e2e["retrieval_generations_run"] = int(sum(lengths))
            e2e["retrieval_generations_full"] = R * cs
            e2e["executed_work_ratio"] = sum(lengths) / (R * cs)
        print(json.dumps({name: walls[name][-1]}), flush=True)
tr.mcmc_get, tr.mcmc_retain = get, retain
for name, v in walls.items():
    e2e[name + "_wall_s"] = dict(runs=v, median=float(np.median(v)), min=min(v), max=max(v))
e2e["wall_ratio_each_over_grtest_only_medians"] = e2e["grexit_each_wall_s"]["median"] / e2e["grtest_only_wall_s"]["median"]
res["end_to_end"] = dict(e2e, chainsize=cs, retrievals=R)
tr.free_memory()
s = json.dumps(res, indent=1, default=str)
if a.out:
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(s + "\n")
print(s)
