#!/usr/bin/env python
"""bench.py -- forward-model spectra/s on the WASP-12b eclipse shape (BASELINE.json metric).

A step = one DE-MC generation on this rank: M proposal models -> spectra -> band fluxes
(atm_prep + fused eclipse column kernel + band integration), plus, for N>1, the per-generation
all-gather of the band fluxes (fused into the band-integration kernel over NVLink peer windows).
`value` is measured with the proposals already resident in HBM; `e2e` goes through the
reference-facing batched call with pinned HOST buffers (profiles H2D, spectra D2H inside the timed
region).  Timing: CUDA events on the library's own stream, max over ranks.

The line proves itself:
  parity       the spectra this run produced for the models the `cpu_baseline` leg also ran
               through the UNMODIFIED reference (oracle/_ref), compared in the run (max relative
               error, last[] identical); above 1e-6 the run fails
  gather_check (N>1) every rank recomputes a sample of every peer's band fluxes and compares them
               with what the fused all-gather delivered
  roofline     the dominant kernel's pipe utilisations and DRAM traffic, measured by an ncu
               subprocess of this run on the same kernel / shape / batch (after the timed region;
               no number printed under ncu is used as a rate)
  hr_lookup    the stand-alone opacity-lookup kernel on a 6.4 GB grid (1e5 wavenumbers), the
               kernel the north star's >=70 % of HBM target is about
  latency      small-population generation latency (10 chains, CUDA-graph replay)
  transit      the transit-geometry configuration (demo BART_transit.cfg shape) on the same GPU
`--impl reference` times the unmodified reference C (oracle/_ref; else the oracle port) on the host
cores for the same configuration.
`--dump-outputs DIR` saves what the last timed step of the device leg and of the two host legs
returned (band fluxes, spectra and status of a seeded sample of the models), so that two builds can
be compared output for output on the same seeded inputs.
"""
import argparse
import csv
import io
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "forward_model_spectra_per_s"
UNIT = "spectra/s"
WORKLOAD = ("WASP-12b eclipse (examples/WASP-12b/BART.cfg shape): 2424 wavenumbers (910-3333 cm-1) "
            "x 100 layers x 27 grid temperatures x 4 molecules (H2O CO2 CO CH4) + H2-H2 CIA, "
            "5 ray angles, toomuch 10, 4 filters")
PARITY_TOL = 1e-6
# --dump-outputs keeps the outputs of this many models, the same seeded sample in every array (~10 MB
# at the W12 shape), and never writes more than DUMP_LIMIT bytes
DUMP_MODELS = 512
DUMP_LIMIT = 64 << 20


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ---------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.proc = None
        self.lines = []

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.lines.append(line.strip())
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); smax.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)),
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------
def make_workload(tmp, rank, M):
    from bart_b200 import synth
    case = synth.make_case(os.path.join(tmp, "w12_rank%d" % rank), shape="w12", solution="eclipse",
                           seed=2026)
    models = synth.make_models(case, M, seed=2026 + rank, molfit=("H2O", "CO2", "CO", "CH4"))
    return case, models


def star_planck(wn, tstar=6300.0):
    hc_k = 6.6260755e-27 * 2.99792458e10 / 1.380658e-16
    return 2 * 6.6260755e-27 * 2.99792458e10 ** 2 * wn ** 3 / np.expm1(hc_k * wn / tstar) * np.pi


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def reference_rate(case, models, nproc, per_proc, timeout=900, want_last=False):
    """Time the CPU implementation of run_transit with `nproc` independent processes (MC3's own
    one-process-per-chain model, mccubed.py:277,393): process p runs models [p per_proc, (p+1) per_proc)
    of the batch.  Returns (models/s, kind, cores, results) where results[p] = (model indices,
    spectra, last|None) as the reference computed them."""
    ref_so = os.path.join(ROOT, "oracle", "_ref", "libtransit_ref.so")
    workdir = case["workdir"]
    results = []
    if os.path.exists(ref_so):
        procs = []
        for p in range(nproc):
            idx = (np.arange(per_proc) + p * per_proc) % len(models)
            mp = os.path.join(workdir, "ref_models_%d.npy" % p)
            np.save(mp, models[idx])
            op = os.path.join(workdir, "ref_out_%d.npz" % p)
            cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_driver.py"), case["cfg"], mp, op,
                   "--time", str(per_proc)] + (["--last"] if want_last else [])
            procs.append((subprocess.Popen(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL), op, idx))
        rate = 0.0
        for pr, op, idx in procs:
            pr.wait(timeout=timeout)
            if pr.returncode == 0 and os.path.exists(op):
                z = np.load(op)
                rate += 1.0 / float(z["sec_per_model"])
                results.append((idx, z["spectra"], z["last"] if "last" in z.files else None))
        return rate, "reference", nproc, results
    # the oracle port (single-threaded restatement), one process
    from oracle import oracle as orc
    O = orc.Oracle(case["cfg"])
    O.run(models[0])
    t0 = time.perf_counter()
    n = min(per_proc, len(models))
    spectra = np.stack([O.run(models[m]) for m in range(n)])
    results.append((np.arange(n), spectra, None))
    return n / (time.perf_counter() - t0), "port", 1, results


def run_reference_arm(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    ncores = os.cpu_count() or 1
    nproc = max(1, min(ncores, 64))
    with tempfile.TemporaryDirectory(prefix="bart_bench_ref_") as tmp:
        case, models = make_workload(tmp, 0, 64)
        per_proc = 6
        for _ in range(args.warmup and 1):
            reference_rate(case, models, nproc, 2)
        t0 = time.perf_counter()
        rates = []
        for _ in range(args.steps):
            r, kind, cores, _ = reference_rate(case, models, nproc, per_proc)
            rates.append(r)
        wall = time.perf_counter() - t0
    value = float(np.mean(rates))
    sample = "%d processes x %d models each per step (run_transit wall time after 2 warm-ups)" % (nproc, per_proc)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * wall / max(1, args.steps), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "models_per_step": nproc * per_proc, "cpu": cpu_model()},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------
NCU_METRICS = ("gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum,"
               "l1tex__data_pipe_lsu_wavefronts.avg.pct_of_peak_sustained_elapsed,"
               "smsp__issue_active.avg.pct_of_peak_sustained_active,"
               "sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active,"
               "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed,"
               "lts__throughput.avg.pct_of_peak_sustained_elapsed,"
               "sm__inst_executed_pipe_fp64.sum,smsp__inst_executed.sum,sm__warps_active.avg.pct_of_peak_sustained_active")


def ncu_measure(cmd, kernel_regex, skip=1, timeout=240):
    """One launch of `kernel_regex` inside `cmd` under ncu (a subprocess of this run, outside every
    timed region): {metric: value}.  None when ncu is not available or fails."""
    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None
    try:
        r = subprocess.run([ncu, "--metrics", NCU_METRICS, "--clock-control", "none", "-k",
                            "regex:" + kernel_regex, "-s", str(skip), "-c", "1", "--csv"] + cmd,
                           capture_output=True, text=True, timeout=timeout)
        rows = [row for row in csv.reader(io.StringIO(r.stdout)) if len(row) > 3]
        hdr = next(row for row in rows if "Metric Name" in row)
        iname, ival, iunit = hdr.index("Metric Name"), hdr.index("Metric Value"), hdr.index("Metric Unit")
        out = {}
        for row in rows[rows.index(hdr) + 1:]:
            try:
                v = float(row[ival].replace(",", ""))
            except ValueError:
                continue
            unit = row[iunit].lower()
            scale = {"kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9, "tbyte": 1e12, "usecond": 1e-3, "us": 1e-3,
                     "msecond": 1.0, "ms": 1.0, "nsecond": 1e-6, "ns": 1e-6, "second": 1e3, "s": 1e3}.get(unit, 1.0)
            out[row[iname]] = v * scale
        return out or None
    except Exception:
        return None


def run_tool(script, extra, timeout=420):
    """A helper of tools/ in its own process (the library holds one configuration per process);
    returns its JSON line or {"error": ...} -- the headline must not depend on it."""
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", script)] + extra,
                           capture_output=True, text=True, timeout=timeout)
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:
        return {"error": repr(e)[:200]}


# ---------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--models", type=int, default=4096, help="proposal models per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU legs (and with them the parity gate)")
    ap.add_argument("--no-extras", action="store_true", help="skip the ncu / hr_lookup / builder / latency legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of each timed leg returned as DIR/<name>.npy "
                         "(float64, for a fixed sample of %d models per rank)" % DUMP_MODELS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    dist = None
    numa_cpus = None
    if world > 1 and os.environ.get("BART_BENCH_NUMA", "1") != "0":
        # one process per GPU: keep each rank (and its pinned host buffers) on its GPU's NUMA node
        from bart_b200 import api as _api
        numa_cpus = _api.bind_to_device_numa(local)
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from bart_b200 import api, synth
    L = api.lib()
    M = args.models
    W = max(3, args.warmup)
    tmp = tempfile.mkdtemp(prefix="bart_bench_")
    case, models = make_workload(tmp, rank, M)
    tr = api.Transit(case["cfg"], device=local)
    info = api.device_info()
    wn = tr.get_waveno_arr()
    start, count, weight, star = api.filters_from_files(wn, case["filters"], wn, star_planck(wn))
    tr.set_filters(start, count, weight, star, 0.117)
    nf, nw, n_in = tr.nfilters, tr.nwave, tr.n_in

    # multi-GPU exchange: library-owned NCCL communicator, unique id through torch.distributed
    if world > 1:
        import ctypes as C
        idbuf = C.create_string_buffer(128)
        if rank == 0:
            api._check(L.bart_comm_unique_id(idbuf))
        obj = [idbuf.raw]
        dist.broadcast_object_list(obj, src=0)
        api._check(L.bart_comm_init(rank, world, obj[0]))

    # device-resident proposals and results
    d_prof = L.bart_dev_alloc(M * n_in * 8)
    d_band = L.bart_dev_alloc(M * nf * 8)
    d_all = L.bart_dev_alloc(world * M * nf * 8)
    api._check(L.bart_memcpy_h2d(d_prof, models.ctypes.data, M * n_in * 8))

    def step_device():
        if world > 1:
            # band integration fused with the all-gather (stores into the peers' NVLink windows;
            # ncclAllGather when the windows could not be mapped)
            api._check(L.bart_bandflux_allgather_device(d_prof, M, n_in, d_band, d_all))
        else:
            api._check(L.bart_bandflux_batch_device(d_prof, M, n_in, d_band, None))

    def barrier():
        L.bart_sync()
        if dist is not None:
            dist.barrier()

    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(W):
        step_device()
    barrier()
    L.bart_profile_reset()
    L.bart_profile_enable(1)
    launches0 = L.bart_launch_count()
    ms = []
    for _ in range(args.steps):
        L.bart_flush_l2()                      # untimed: evict the L2 between steps
        barrier()
        L.bart_timer_begin()
        step_device()
        ms.append(L.bart_timer_end())
    barrier()
    launches = L.bart_launch_count() - launches0                   # L2-flush fills are not counted
    L.bart_profile_enable(0)
    stats = api.kernel_stats()
    total_ms = float(np.sum(ms))
    # --dump-outputs: the band fluxes of the last timed step (the gathered blocks of every rank for N>1,
    # rank after rank), read before any later leg reuses the buffers
    dumps = {}
    if args.dump_outputs:
        dump_rows = np.sort(np.random.default_rng(0).choice(M, min(M, DUMP_MODELS), replace=False))
        band = np.empty((world, M, nf))
        api._check(L.bart_memcpy_d2h(band.ctypes.data, d_all if world > 1 else d_band, band.nbytes))
        dumps["band_flux"] = band[:, dump_rows].reshape(-1, nf)

    # N>1: what the fused all-gather delivered, against a local recompute of a sample of every
    # rank's models (each rank's batch is seeded by its rank, so any rank can rebuild it)
    gather = None
    if world > 1:
        nchk = min(64, M)
        got = np.empty((world, M, nf))
        api._check(L.bart_memcpy_d2h(got.ctypes.data, d_all, world * M * nf * 8))
        worst, bad = 0.0, 0
        for q in range(world):
            mq = models if q == rank else synth.make_models(case, M, seed=2026 + q,
                                                            molfit=("H2O", "CO2", "CO", "CH4"))
            ref, _ = tr.bandflux_batch(mq[:nchk])
            d = np.abs(got[q, :nchk] - ref)
            worst = max(worst, float(d.max()))
            bad += int((got[q, :nchk] != ref).sum())
        own = np.empty((M, nf))
        api._check(L.bart_memcpy_d2h(own.ctypes.data, d_band, M * nf * 8))
        bad += int((got[rank] != own).sum())
        gather = {"max_abs_diff": worst, "mismatches": bad}

    # end to end through the reference-facing batched call: pinned host in/out
    h_in = api.PinnedArray((M, n_in))
    h_out = api.PinnedArray((M, nw))
    h_band = api.PinnedArray((M, nf))
    h_in.array[:] = models
    st = np.zeros(M, dtype=np.int32)
    for _ in range(2):
        tr.run_batch(h_in.array, out=h_out.array, status=st)
    e2e_ms = []
    for _ in range(args.steps):
        L.bart_flush_l2()
        barrier()
        t0 = time.perf_counter()
        tr.run_batch(h_in.array, out=h_out.array, status=st)
        e2e_ms.append(1e3 * (time.perf_counter() - t0))
    e2e_total = float(np.sum(e2e_ms))
    if args.dump_outputs:
        dumps["e2e_spectra"] = h_out.array[dump_rows]
        dumps["e2e_status"] = st[dump_rows]
    # the same, returning what BART consumes (band fluxes, BARTfunc.py:386-399) instead of spectra
    for _ in range(2):
        tr.bandflux_batch(h_in.array, out=h_band.array, status=st)
    e2b_ms = []
    for _ in range(args.steps):
        L.bart_flush_l2()
        barrier()
        t0 = time.perf_counter()
        tr.bandflux_batch(h_in.array, out=h_band.array, status=st)
        e2b_ms.append(1e3 * (time.perf_counter() - t0))
    e2b_total = float(np.sum(e2b_ms))
    if args.dump_outputs:
        dumps["e2e_band_flux"] = h_band.array[dump_rows]
        dumps["e2e_band_status"] = st[dump_rows]
    # nvidia-smi can take longer to start than a short run lasts (8 ranks on one box): keep the
    # same step running, untimed, until the sampler has seen the GPU under this load
    t_wait = time.time()
    while len(sampler.lines) < 5 and time.time() - t_wait < 8.0:
        # rank-local work only: the number of iterations differs between ranks
        api._check(L.bart_bandflux_batch_device(d_prof, M, n_in, d_band, None))
    clocks = sampler.stop()

    if dist is not None:
        import torch
        t = torch.tensor([total_ms, e2e_total, e2b_total,
                          gather["max_abs_diff"], float(gather["mismatches"])], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_total, e2b_total = float(t[0]), float(t[1]), float(t[2])
        gather = {"ranks": world, "models_checked_per_peer": min(64, M), "max_abs_diff": float(t[3]),
                  "mismatches_max_over_ranks": int(t[4]), "ok": bool(t[4] == 0),
                  "what": "band fluxes delivered by the fused all-gather vs a local recompute of every "
                          "peer's first models (bit-exact expected), and the own block vs the local result"}

    rc = 0
    if rank == 0:
        value = world * M * args.steps / (total_ms * 1e-3)
        e2e_value = world * M * args.steps / (e2e_total * 1e-3)
        e2b_value = world * M * args.steps / (e2b_total * 1e-3)
        nmol, nlayer = L.bart_ngridmol(), tr.nlayer
        alg_bytes = M * (16.0 * nmol * nlayer * nw + 8.0 * nw)
        dom = "eclipse_column"
        k = stats.get(dom, {"launches": 0, "ms": 0.0})
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        try:
            peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
            peak_src = "MEASURED_PEAKS.json"
        except Exception:
            pass
        k_ms = (k["ms"] / k["launches"]) if k["launches"] else None
        hbm_alg = alg_bytes / (k_ms * 1e-3) / 1e9 if k_ms else None

        extras = world == 1 and not args.no_extras
        # --- the dominant kernel under ncu, in this run (same shape, same batch size)
        prof = None
        if extras:
            prof = ncu_measure([sys.executable, os.path.join(ROOT, "tools", "profile_step.py"),
                                "--models", str(M), "--steps", "2"], "eclipse_column_kernel")
        pipes, traffic, src = None, None, None
        if prof:
            pipes = {"l1_data_pipe": prof.get("l1tex__data_pipe_lsu_wavefronts.avg.pct_of_peak_sustained_elapsed", 0) / 100,
                     "issue_slots": prof.get("smsp__issue_active.avg.pct_of_peak_sustained_active", 0) / 100,
                     "fp64_pipe": prof.get("sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active", 0) / 100,
                     "l2": prof.get("lts__throughput.avg.pct_of_peak_sustained_elapsed", 0) / 100,
                     "dram": prof.get("gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", 0) / 100,
                     "warps_active": prof.get("sm__warps_active.avg.pct_of_peak_sustained_active", 0) / 100}
            traffic = prof.get("dram__bytes_read.sum", 0.0) + prof.get("dram__bytes_write.sum", 0.0)
            src = "ncu subprocess of this run (one launch, %d models)" % M
        else:
            try:
                pj = json.load(open(os.path.join(ROOT, "profiles", "eclipse_column_pipes.json")))
                if pj.get("models_per_launch") == M:
                    pipes, traffic = pj["pipes"], pj.get("dram_bytes_per_launch")
                    src = "profiles/eclipse_column_pipes.json (ncu not run in this invocation)"
            except Exception:
                pass
        # The kernel is not HBM-bound at this shape (the 209 MB grid is served from L2; DRAM a few % of
        # peak): what bounds it is the SM -- L1 data pipe (grid samples + table records + exp
        # tables), issue slots and the fp64 pipe, in that order.  `frac` is the busiest of them.
        top = max(((v, n) for n, v in pipes.items() if n in ("l1_data_pipe", "issue_slots", "fp64_pipe")),
                  default=(None, None)) if pipes else (None, None)
        clock_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
        fp64_inst = prof.get("sm__inst_executed_pipe_fp64.sum") if prof else None
        roofline = {"kernel": dom, "bound": "sm:" + top[1] if top[1] else "sm",
                    "achieved": top[0] * 100 if top[0] is not None else None, "peak": 100.0,
                    "unit": "% of pipe peak", "frac": top[0], "pipes": pipes, "pipes_source": src,
                    "traffic": traffic,
                    "fp64": {"warp_instructions_per_launch": fp64_inst,
                             "frac_of_peak_from_counts": (fp64_inst * 2.0 / (info["sm_count"] * 4 * clock_hz * k_ms * 1e-3))
                             if fp64_inst and k_ms else None,
                             "peak": "1 warp DFMA per 2 cycles per SM sub-partition (64 lanes/clk/SM), at the SM "
                                     "clock sampled under load"},
                    "hbm_algorithmic": {"achieved": hbm_alg, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                                        "frac": (hbm_alg / peak) if hbm_alg else None,
                                        "algorithmic_bytes_per_launch": alg_bytes,
                                        "note": "SURVEY 8(d) accounting (two bracketing planes per layer per model, no "
                                                "credit for the toomuch early exit or cache reuse): served from L2, "
                                                "so > 1 is reuse, not HBM bandwidth"},
                    "kernel_ms_per_launch": k_ms,
                    "kernel_share_of_step": (k["ms"] / total_ms) if total_ms else None}

        # --- CPU legs: the unmodified reference on the host cores + the in-run parity gate
        cpu, parity = None, None
        if world == 1 and not args.no_cpu_baseline:
            ncores = os.cpu_count() or 1
            nproc = max(1, min(ncores, 64))
            r1, kind1, _, _ = reference_rate(case, models, 1, 6)
            rate, kind, cores, results = reference_rate(case, models, nproc, 6, want_last=True)
            cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": kind, "cpu": cpu_model(),
                   "single_thread_value": r1,
                   "sample": "%d processes x 6 models of the same batch (run_transit wall time after 2 "
                             "warm-ups; reference writes its output spectrum to /dev/null); "
                             "single_thread_value: one process alone on the box" % nproc}
            # parity: the production kernel's spectra of exactly those models (h_out holds the whole
            # batch from the e2e leg) and, through the introspection kernel, last[]
            worst, nmod, last_ok, nlast = 0.0, 0, True, 0
            for idx, ref_spec, ref_last in results:
                gpu_spec = h_out.array[idx]
                worst = max(worst, float(np.max(np.abs(gpu_spec - ref_spec) / np.abs(ref_spec))))
                nmod += len(idx)
                if ref_last is not None:
                    tr.debug_keep(True)
                    tr.run_batch(models[idx])
                    for j in range(len(idx)):
                        gl = tr.debug_get("last", j).astype(np.int64)
                        last_ok = last_ok and bool(np.array_equal(gl, ref_last[j]))
                        nlast += 1
                    tr.debug_keep(False)
            parity = {"vs": "unmodified reference (oracle/_ref)" if kind == "reference" else "oracle port",
                      "n_models": nmod, "max_rel_err": worst, "last_identical": last_ok if nlast else None,
                      "n_models_last": nlast, "tol": PARITY_TOL, "ok": bool(worst <= PARITY_TOL and last_ok)}
            if not parity["ok"]:
                rc = 1

        hr, builder, latency, transit = None, None, None, None
        if extras:
            # the kernel the north star's ">= 70 % of HBM" target is meaningful for: the stand-alone
            # lookup on a grid far larger than the L2 (1e5 wavenumbers, 6.4 GB), one model per launch
            hr = run_tool("bench_lookup.py", ["--models", "1,4", "--fused-models", "64", "--steps", "5"])
            b = run_tool("bench_builder.py", [], timeout=300)
            if "error" in b:
                builder = b
            else:
                builder = {"metric": "opacity_grid_builder_line_cells_per_s",
                           "value": b["line_cells_per_s_device"], "unit": "lines x (T,layer) cells / s",
                           "wall_value": b["line_cells_per_s_wall"],
                           "sample": "%d synthetic lines x %d layers x %d temperature planes on the W12 "
                                     "wavenumber grid (%d samples, wnosamp %d)" % (
                                         b["nlines_in_range"], b["shape"]["nlayer"], b["shape"]["ntemp_built"],
                                         b["shape"]["nwave"], b["shape"]["wnosamp"]),
                           "per_slice_ms": b["per_slice_ms"]}
            latency = run_tool("bench_latency.py", [])
            transit = run_tool("bench_transit.py", [])

        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": W, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": WORKLOAD, "models_per_gpu_per_step": M,
                           "parallelism": "chains partitioned by rank (dp%d); per-generation all-gather "
                                          "of band fluxes %s" % (world, "fused into the band-integration "
                                          "kernel (stores into peer windows over NVLink)"
                                          if world > 1 and L.bart_comm_p2p() else "(ncclAllGather)"
                                          if world > 1 else "(single rank: none)"),
                           "l2": "flushed between steps (256 MB write); grid 209 MB > L2",
                           "device": info["name"], "sm_count": info["sm_count"]},
                "roofline": roofline, "cpu_baseline": cpu, "parity": parity,
                "numa_bound_cpus_rank0": (len(numa_cpus) if numa_cpus else None),
                # what a BART worker hands to MC3 per proposal is the band fluxes (BARTfunc.py:386-399):
                # host profiles in, band fluxes out is the end-to-end unit of the retrieval loop
                "e2e": {"value": e2b_value, "unit": UNIT, "h2d_bytes_per_step": M * n_in * 8,
                        "d2h_bytes_per_step": M * nf * 8 + M * 4,
                        "path": "bart_bandflux_batch: pinned host profiles -> H2D -> kernels (forward model + "
                                "band integration) -> D2H band fluxes + status, i.e. run_transit + "
                                "BARTfunc.py:386-399 for a batch of proposals"},
                # the same with the full spectra returned to the host (batched run_transit, 19 KB per
                # model): at N = 8 this leg is bound by the host's memory system, not by the GPUs
                "e2e_spectra": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": M * n_in * 8,
                                "d2h_bytes_per_step": M * nw * 8 + M * 4,
                                "path": "bart_run_batch: pinned host profiles -> H2D -> kernels -> D2H spectra"},
                "gpu_launches": int(launches), "kernels": stats, "clocks": clocks}
        if gather is not None:
            line["gather_check"] = gather
            if not gather["ok"]:
                rc = 1
        if hr is not None:
            line["hr_lookup"] = hr
        if builder is not None:
            line["builder"] = builder
        if latency is not None:
            line["latency"] = latency
        if transit is not None:
            line["transit"] = transit
        if rc:
            line["valid"] = False
        if args.dump_outputs:
            out = {name: np.ascontiguousarray(a, dtype=np.float64) for name, a in dumps.items()}
            assert sum(a.nbytes for a in out.values()) <= DUMP_LIMIT, "--dump-outputs over %d bytes" % DUMP_LIMIT
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in out.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line))
    if dist is not None:
        L.bart_comm_finalize()
        dist.destroy_process_group()
    return rc


if __name__ == "__main__":
    sys.exit(main() or 0)
