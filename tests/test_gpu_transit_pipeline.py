"""GPU: the transit tile kernels' chunk pipeline with the chord weights staged by bulk-async copy
(TMA) and by the plain cooperative copy.

Both the tensor-core (DMMA) kernel and the DFMA tile kernel copy each depth chunk's weights into
shared memory while the previous chunk is scanned.  The two staging forms must give bit-identical
spectra and status words in each kernel, within TIGHT of the oracle, and the introspection launch
must stop at the oracle's last[] under either form.  The cases cover the transmission scan
(`tiny_transit`), the scattering / cloud build (`small4_transit_cloud`) and modlevel -1
(`tiny_transit_m1`).  BART_NO_TMA is read once when the device is opened, so the plain form runs in
a subprocess."""
import os
import subprocess
import sys

import numpy as np
import pytest

import cases
from util import relerr, apply_setters

pytestmark = pytest.mark.gpu
TIGHT = 1e-8
CASES = ["tiny_transit", "small4_transit_cloud", "tiny_transit_m1"]
KERNELS = {"default": None, "dfma": "0"}       # -> BART_TRANSIT_MMA


def run_kernels(cfg, models, setters):
    """Spectra and status of each kernel choice, and last[] of the introspection launch."""
    from bart_b200 import api
    tr = api.Transit(cfg)
    apply_setters(tr, setters)
    out = {}
    for name, mma in KERNELS.items():
        if mma is None:
            os.environ.pop("BART_TRANSIT_MMA", None)
        else:
            os.environ["BART_TRANSIT_MMA"] = mma
        out[name + "_spectra"], out[name + "_status"] = tr.run_batch(models)
    os.environ.pop("BART_TRANSIT_MMA", None)
    tr.debug_keep(True)
    tr.run_batch(models)
    out["last"] = np.stack([tr.debug_get("last", m).astype(np.int64) for m in range(models.shape[0])])
    tr.free_memory()
    return out


@pytest.fixture(scope="module")
def api(built):
    from bart_b200 import api as a
    info = a.device_info()
    assert info["cc"][0] >= 10, info
    return a


@pytest.mark.parametrize("name", CASES)
def test_tma_and_plain_weight_staging_agree(name, api, get_case, monkeypatch):
    from oracle import oracle as orc
    case, models, setters = get_case(name)
    monkeypatch.delenv("BART_TRANSIT_MMA", raising=False)
    tma = run_kernels(case["cfg"], models, setters)
    mp = os.path.join(case["workdir"], "m_pipe.npy")
    op = os.path.join(case["workdir"], "o_pipe.npz")
    np.save(mp, models)
    code = ("import sys, numpy as np; sys.path[:0] = [%r, %r]; import test_gpu_transit_pipeline as t; "
            "np.savez(%r, **t.run_kernels(%r, np.load(%r), %r))"
            % (cases.ROOT, os.path.join(cases.ROOT, "tests"), op, case["cfg"], mp, setters))
    env = dict(os.environ, BART_NO_TMA="1")
    env.pop("BART_TRANSIT_MMA", None)
    subprocess.check_call([sys.executable, "-c", code], env=env)
    plain = dict(np.load(op))
    O = orc.Oracle(case["cfg"])
    apply_setters(O, setters)
    ref = [O.run(models[m], inter=True) for m in range(models.shape[0])]
    for k in KERNELS:
        assert np.array_equal(plain[k + "_spectra"], tma[k + "_spectra"]), k
        assert np.array_equal(plain[k + "_status"], tma[k + "_status"]), k
        assert (tma[k + "_status"] == 0).all(), k
        for m, o in enumerate(ref):
            assert relerr(tma[k + "_spectra"][m], o["spectrum"]) < TIGHT, (k, m)
    for last in (tma["last"], plain["last"]):
        for m, o in enumerate(ref):
            assert np.array_equal(last[m], o["last"]), m
