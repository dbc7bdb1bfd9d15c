"""Worker of tests/test_gpu_mcmc_device_draws.py: one process per GPU (rank = argv[1]) running seeded
DE-MC and snooker ensembles (streams drawn on every rank from the same Philox keys) whose flattened
population is split over the ranks.  `run_seeded_ensembles` is also the single-GPU run the test
compares against."""
import os
import sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

from ensemble_rank_worker import NAME, NRETR, make_transit  # noqa: E402

KEYS = [(1000 + r, 0xA5A5A5A5A5A5A5A5) for r in range(NRETR)]


def run_seeded_ensembles(api, workdir, device=None, tr=None):
    import cases
    from bart_b200 import driver
    spec = cases.RETRIEVAL[NAME]
    if tr is None:
        tr, spec = make_transit(api, workdir, device)
    d = np.load(os.path.join(cases.GOLDEN_DIR, "retrieval_mc3_%s.npz" % NAME))
    data = np.array([d["data"] * (1 + 0.01 * np.random.RandomState(900 + r).normal(size=len(d["data"])))
                     for r in range(NRETR)])
    uncert = np.repeat(d["uncert"][None], NRETR, 0)
    args = (spec["pmin"], spec["pmax"], spec["stepsize"], spec["numit"], spec["nchains"])
    rngs = lambda: [np.random.RandomState(41 + r) for r in range(NRETR)]
    keys = ("allparams", "allmodel", "params", "numaccept", "outbounds", "bestp", "bestchisq",
            "bestmodel", "currchisq", "models")
    res = {}
    outs = driver.run_demc_ensemble(tr, data, uncert, [spec["params"]] * NRETR, *args, burnin=spec["burnin"],
                                    rngs=rngs(), seeds=KEYS)
    res.update({"demc_" + k: np.stack([np.asarray(o[k]) for o in outs]) for k in keys})
    outs = driver.run_snooker_ensemble(tr, data, uncert, [spec["params"]] * NRETR, *args, burnin=spec["burnin"],
                                       thinning=2, rngs=rngs(), seeds=KEYS)
    res.update({"snooker_" + k: np.stack([np.asarray(o[k]) for o in outs]) for k in keys + ("Z", "Zchisq")})
    tr.free_memory()
    return res


def main():
    rank, world, workdir, outpath = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], sys.argv[4]
    import ctypes as C
    import time
    from bart_b200 import api
    L = api.lib()
    tr, spec = make_transit(api, os.path.join(workdir, "rank%d" % rank), rank)
    idfile = os.path.join(workdir, "nccl_id_seeded.bin")
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
    res = run_seeded_ensembles(api, workdir, tr=tr)
    np.savez(outpath, p2p=p2p, **res)
    L.bart_comm_finalize()


if __name__ == "__main__":
    main()
