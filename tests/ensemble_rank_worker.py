"""Worker of tests/test_gpu_retrieval_ensemble.py: one process per GPU (rank = argv[1]) running a
4-retrieval DE-MC ensemble whose flattened population is split over the ranks; NCCL unique id
exchanged through a file.  `run_ensemble` is also the single-GPU run the test compares against."""
import os
import sys
import time
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

NAME, NRETR = "retr_tiny_eclipse", 4


def make_transit(api, workdir, device):
    import cases
    case, spec, extra = cases.build_retrieval(NAME, workdir)
    tr = api.Transit(case["cfg"], device=device)
    wn = tr.get_waveno_arr()
    start, count, weight, star = api.filters_from_files(wn, case["filters"], extra["starwn"], extra["starfl"])
    tr.set_filters(start, count, weight, star, extra["rprs"])
    tr.converter_init(case["press_bar"], case["species"], case["abund"], spec["molfit"], spec["pt"],
                      pt_args=extra["pt_args"], nrad=spec["nrad"], ncloud=spec["ncloud"], nray=spec["nray"])
    return tr, spec


def run_ensemble(api, workdir, device=None, tr=None):
    """The ensemble both sides run: golden data plus seeded noise per retrieval, start points and
    streams from RandomState(31 + r).  Returns its arrays stacked over the retrievals."""
    import cases
    from bart_b200 import driver
    spec = cases.RETRIEVAL[NAME]
    if tr is None:
        tr, spec = make_transit(api, workdir, device)
    d = np.load(os.path.join(cases.GOLDEN_DIR, "retrieval_mc3_%s.npz" % NAME))
    data = np.array([d["data"] * (1 + 0.01 * np.random.RandomState(900 + r).normal(size=len(d["data"])))
                     for r in range(NRETR)])
    uncert = np.repeat(d["uncert"][None], NRETR, 0)
    outs = driver.run_demc_ensemble(tr, data, uncert, [spec["params"]] * NRETR, spec["pmin"], spec["pmax"],
                                    spec["stepsize"], spec["numit"], spec["nchains"], burnin=spec["burnin"],
                                    rngs=[np.random.RandomState(31 + r) for r in range(NRETR)])
    keys = ("allparams", "allmodel", "params", "numaccept", "outbounds", "bestp", "bestchisq",
            "bestmodel", "currchisq", "models")
    res = {k: np.stack([np.asarray(o[k]) for o in outs]) for k in keys}
    tr.free_memory()
    return res


def main():
    rank, world, workdir, outpath = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3], sys.argv[4]
    import ctypes as C
    from bart_b200 import api
    L = api.lib()
    tr, spec = make_transit(api, os.path.join(workdir, "rank%d" % rank), rank)
    idfile = os.path.join(workdir, "nccl_id_ensemble.bin")
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
    lo, hi = C.c_int(), C.c_int()
    L.bart_chain_block(NRETR * spec["nchains"], world, rank, C.byref(lo), C.byref(hi))
    assert 0 < hi.value - lo.value < NRETR * spec["nchains"]
    res = run_ensemble(api, workdir, tr=tr)
    np.savez(outpath, p2p=p2p, **res)
    L.bart_comm_finalize()


if __name__ == "__main__":
    main()
