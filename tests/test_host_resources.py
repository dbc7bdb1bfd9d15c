"""Host resources of libbart_b200: device buffers, pinned buffers and file handles are held by
owning types (bart_b200/csrc/cuda_host.hpp; the file owners in host.hpp, which the CUDA-free
emulation build of readers.cpp includes too), so that free_memory and a fail() on an error path
leave nothing behind.
CPU: no raw allocation or open/close outside those owners, the C-ABI pass-through allocators and
the peer window's CUDA IPC mappings.
GPU: free device memory and the open file descriptors come back to where they were after
configurations that end normally and after transit_init calls that fail on malformed input files
(error mode 1: fail() throws)."""
import os
import re
import shutil
import numpy as np
import pytest

import cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "bart_b200", "csrc")

CUDA_NAMES = ("cudaMalloc", "cudaFree", "cudaMallocHost", "cudaFreeHost")
FILE_NAMES = ("fopen", "open(", "close(")
OWNERS = {"cuda_host.hpp": CUDA_NAMES + FILE_NAMES, "host.hpp": FILE_NAMES}
# functions whose raw calls are their contract: memory handed to the caller, CUDA IPC peer windows
RAW_FUNCTIONS = ("bart_dev_alloc", "bart_dev_free", "bart_host_alloc_pinned", "bart_host_free_pinned",
                 "setup_peer_window", "release_peer_window")


def _strip_comments(src):
    src = re.sub(r"/\*.*?\*/", lambda m: "\n" * m.group(0).count("\n"), src, flags=re.S)
    return re.sub(r"//[^\n]*", "", src)


def _blank_function(src, name):
    """src with the body of every definition of `name` blanked (line numbers kept)."""
    for m in list(re.finditer(r"^[A-Za-z][^;{}()]*\b%s\s*\([^;{]*\{" % name, src, flags=re.M))[::-1]:
        depth, i = 1, m.end()
        while depth:
            depth += {"{": 1, "}": -1}.get(src[i], 0)
            i += 1
        body = src[m.start():i]
        src = src[:m.start()] + re.sub(r"[^\n]", " ", body) + src[i:]
    return src


def _pattern(name):
    return r"\b" + re.escape(name) + ("" if name.endswith("(") else r"\b")


def test_resources_only_through_owners():
    sources = [f for f in sorted(os.listdir(CSRC))
               if f.endswith((".cu", ".cpp", ".hpp", ".cuh", ".h", ".inc"))]
    assert "transit.cu" in sources and "cuda_host.hpp" in sources
    found = []
    for f in sources:
        src = _strip_comments(open(os.path.join(CSRC, f)).read())
        for fn in RAW_FUNCTIONS:
            src = _blank_function(src, fn)
        for name in CUDA_NAMES + FILE_NAMES:
            if name in OWNERS.get(f, ()):
                continue
            for m in re.finditer(_pattern(name), src):
                found.append("%s:%d: %s" % (f, src.count("\n", 0, m.start()) + 1, name))
        for name in ("d_mcd", "d_mci"):
            if re.search(r"\b%s\b" % name, src):
                found.append("%s: %s" % (f, name))
    assert not found, "raw resource calls outside the owners:\n" + "\n".join(found)


def test_raw_function_bodies_are_found():
    """The exemption above blanks real function bodies (a renamed function would exempt nothing)."""
    src = _strip_comments(open(os.path.join(CSRC, "transit.cu")).read())
    for fn in RAW_FUNCTIONS:
        blanked = _blank_function(src, fn)
        assert blanked != src and len(blanked) == len(src), fn


# ---------------------------------------------------------------------------------------
# GPU
def _free_bytes():
    import torch
    return torch.cuda.mem_get_info()[0]


def _nfds():
    return len(os.listdir("/proc/self/fd"))


def _grid_mcmc(api, workdir):
    case, spec, extra = cases.build_retrieval("retr_tiny_eclipse", workdir)
    tr = api.Transit(case["cfg"])
    wn = tr.get_waveno_arr()
    start, count, weight, star = api.filters_from_files(wn, case["filters"], extra["starwn"], extra["starfl"])
    tr.set_filters(start, count, weight, star, extra["rprs"])
    tr.converter_init(case["press_bar"], case["species"], case["abund"], spec["molfit"], spec["pt"],
                      pt_args=extra["pt_args"], nrad=spec["nrad"], ncloud=spec["ncloud"], nray=spec["nray"])
    nch = spec["nchains"]
    stepsize = np.array(spec["stepsize"])
    ifree = stepsize > 0
    rng = np.random.RandomState(3)
    p0 = np.repeat(np.atleast_2d(spec["params"]), nch, 0)
    p0[:, ifree] += rng.normal(0, 0.01, (nch, int(ifree.sum())))
    nf = len(case["filters"])
    tr.mcmc_init(p0, spec["pmin"], spec["pmax"], stepsize, np.ones(nf), np.full(nf, 0.1))
    pmin, pmax = np.array(spec["pmin"])[ifree], np.array(spec["pmax"])[ifree]
    tr.mcmc_snooker_init(rng.uniform(pmin, pmax, (nch + 1, nch, int(ifree.sum()))), 1)
    tr.free_memory()


def _just_opacity(api, workdir):
    case = cases.build_builder_case("build_ch4", workdir)
    tr = api.Transit(argv=["transit", "-c", case["cfg"], "--justOpacity"])
    assert os.path.getsize(case["opacity"]) > 0
    tr.free_memory()


def _lbl_batch(api, workdir):
    case, models = cases.build_lbl_case("lbl_eclipse", workdir)
    tr = api.Transit(case["cfg"])
    spectra, status = tr.run_batch(models)
    assert np.isfinite(spectra).all()
    tr.free_memory()


def _failing_init(api, cfg, match):
    with pytest.raises(api.BartError, match=match):
        api.Transit(cfg)
    api.lib().free_memory()


def _truncated_grid(api, workdir):
    from bart_b200 import synth
    case = synth.make_case(os.path.join(workdir, "res_trunc_grid"), shape="tiny", nlayer=20, seed=81)
    size = os.path.getsize(case["opacity"])
    with open(case["opacity"], "r+b") as f:
        f.truncate(size - size // 3)                    # inside the grid data, past the header
    _failing_init(api, case["cfg"], "truncated")


def _truncated_tli_header(api, workdir):
    from bart_b200 import synth
    case = synth.make_case(os.path.join(workdir, "res_trunc_tli"), shape="tiny", nlayer=20, seed=82)
    with open(case["tli"], "r+b") as f:
        f.truncate(30)                                  # inside the first database name
    _failing_init(api, case["cfg"], "end of file")


def _ungrouped_lines(api, workdir):
    """Line-by-line init whose isotope column is not sorted: the device grouping refuses it."""
    src = cases.build_lbl_case("lbl_eclipse", workdir)[0]
    dst = os.path.join(workdir, "res_ungrouped")
    shutil.rmtree(dst, ignore_errors=True)
    shutil.copytree(src["workdir"], dst)
    tli = os.path.join(dst, os.path.basename(src["tli"]))
    n = len(src["lines"]["isoid"])
    size = os.path.getsize(tli)
    with open(tli, "r+b") as f:                         # columns wl[n] iso[n] elow[n] gf[n] at the end
        f.seek(size - 18 * n)
        f.write(np.ascontiguousarray(src["lines"]["isoid"][::-1]).astype("<i2").tobytes())
    cfg = open(src["cfg"]).read().replace(src["workdir"], dst)
    with open(os.path.join(dst, "transit.cfg"), "w") as f:
        f.write(cfg)
    _failing_init(api, os.path.join(dst, "transit.cfg"), "not grouped by isotope")


CYCLES = {"grid_mcmc_snooker": _grid_mcmc, "just_opacity": _just_opacity, "lbl_batch": _lbl_batch,
          "truncated_grid": _truncated_grid, "truncated_tli_header": _truncated_tli_header,
          "ungrouped_lines": _ungrouped_lines}


@pytest.fixture(scope="module")
def baseline(built, workdir):
    from bart_b200 import api, synth
    case = synth.make_case(os.path.join(workdir, "res_base"), shape="tiny", nlayer=20, seed=80)
    api.Transit(case["cfg"]).free_memory()
    _free_bytes()                                       # torch's CUDA start-up opens descriptors
    return api, _nfds()


@pytest.mark.gpu
@pytest.mark.parametrize("cycle", list(CYCLES))
def test_cycle_returns_memory_and_handles(cycle, baseline, workdir):
    """The first run pays the one-time costs (kernels loaded on first use); a second identical run
    must then leave free device memory where the first left it, within one 2 MiB granule."""
    api, fds = baseline
    CYCLES[cycle](api, workdir)
    assert _nfds() == fds
    free = _free_bytes()
    CYCLES[cycle](api, workdir)
    assert _nfds() == fds
    assert _free_bytes() >= free - (2 << 20), "device memory not returned by %s" % cycle
