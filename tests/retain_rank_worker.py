"""Worker of tests/test_gpu_ensemble_retire.py: one process per GPU (rank = argv[1]) running a
4-retrieval DE-MC ensemble retained to 3 and then to 1 retrieval, so the flattened population
split over the ranks goes 24 -> 18 -> 6 models; NCCL unique id exchanged through a file.
`run_sequence` is also the single-GPU run the test compares against."""
import os
import sys
import time
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

from ensemble_rank_worker import NAME, NRETR, make_transit  # noqa: E402


def run_sequence(api, workdir, device=None, tr=None):
    """Golden data plus seeded noise per retrieval, streams from RandomState(41 + r); 8
    generations, retain [0, 1, 3], 8 more, retain [1] (old retrieval 1), 8 more.  Returns the
    traces of every call and the state after each retain, keyed by step."""
    import cases
    from bart_b200 import driver
    spec = cases.RETRIEVAL[NAME]
    if tr is None:
        tr, spec = make_transit(api, workdir, device)
    d = np.load(os.path.join(cases.GOLDEN_DIR, "retrieval_mc3_%s.npz" % NAME))
    nch, n = spec["nchains"], 8
    step = np.array(spec["stepsize"], dtype=float)
    data = np.array([d["data"] * (1 + 0.01 * np.random.RandomState(900 + r).normal(size=len(d["data"])))
                     for r in range(NRETR)])
    uncert = np.repeat(d["uncert"][None], NRETR, 0)
    rngs = [np.random.RandomState(41 + r) for r in range(NRETR)]
    starts = np.array([driver.start_points(spec["params"], nch, step, np.array(spec["pmin"]),
                                           np.array(spec["pmax"]), g) for g in rngs])
    draws = [driver.demc_draws(g, nch, 3 * n, step[step > 0]) for g in rngs]
    tr.mcmc_init_ensemble(starts, spec["pmin"], spec["pmax"], step, data, uncert, burnin=2)
    res, live = {}, list(range(NRETR))
    for k, keep in enumerate(([0, 1, 3], [1], None)):
        tr.mcmc_run(*driver.stack_demc_draws([draws[r] for r in live], k * n, (k + 1) * n))
        for name in ("allparams", "allmodel", "models", "params", "numaccept", "bestp", "bestchisq"):
            res["%s_%d" % (name, k)] = tr.mcmc_get(name)
        if keep:
            tr.mcmc_retain(keep)
            live = [live[j] for j in keep]
    tr.free_memory()
    return res


def main():
    rank, world, workdir, outpath = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], sys.argv[4]
    import ctypes as C
    from bart_b200 import api
    L = api.lib()
    tr, spec = make_transit(api, os.path.join(workdir, "rank%d" % rank), rank)
    idfile = os.path.join(workdir, "nccl_id_retain.bin")
    if rank == 0:
        buf = C.create_string_buffer(128)
        api._check(L.bart_comm_unique_id(buf))
        with open(idfile + ".tmp", "wb") as f:
            f.write(buf.raw)
        os.rename(idfile + ".tmp", idfile)
    t0 = time.time()
    while not os.path.exists(idfile):
        if time.time() - t0 > 60:
            raise SystemExit("no NCCL id")
        time.sleep(0.05)
    with open(idfile, "rb") as f:
        uid = f.read()
    api._check(L.bart_comm_init(rank, world, uid))
    p2p = L.bart_comm_p2p()
    res = run_sequence(api, workdir, tr=tr)
    np.savez(outpath, p2p=p2p, **res)
    L.bart_comm_finalize()


if __name__ == "__main__":
    main()
