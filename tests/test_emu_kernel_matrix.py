"""CPU: the eclipse throughput kernel's template sets, run on the host by tests/cpu_emu
(emu_run_build), against the oracle.

The emulator selects the build as launch_eclipse does: the specialised (grid molecules, CIA files)
pair with the default ray grid by squaring or a run-time angle count, with or without the
scattering / cloud terms, two columns 64 samples apart per thread with the Planck chaining; and the
run-time-count build with the generic Planck term otherwise.  Both load orders of the specialised
builds (one depth ahead, in step) must give the same bits.  The configurations are those of
tests/test_gpu_kernel_matrix.py, which runs the same builds on the device."""
import numpy as np
import pytest

from emu import Emu
from test_gpu_kernel_matrix import (ECL_PARAMS, ECL_SETTERS, matrix_case, oracle_refs,
                                    expected_status, wide_planck_case)
from util import relerr, apply_setters

PARAMS = ECL_PARAMS + [("wide", "planck", None)]


def expected_build(nmol, ncia):
    return (nmol, ncia) if nmol <= 4 and ncia <= 2 else (0, -1)


@pytest.mark.parametrize("nmol,ncia,raygrid", PARAMS,
                         ids=["%s-%s%s" % ("%dmol" % n if n != "wide" else n, "%dcia" % k if k != "planck" else k,
                                           "-3ang" if r else "") for n, k, r in PARAMS])
def test_throughput_builds_on_the_host(nmol, ncia, raygrid, built, workdir):
    if nmol == "wide":
        case, models = wide_planck_case(workdir)
        build, status = (0, -1), np.zeros(3, dtype=np.int32)
    else:
        case, models = matrix_case(workdir, nmol, ncia, raygrid=raygrid)
        build, status = expected_build(nmol, ncia), expected_status(ncia)
    E = Emu(case["cfg"])
    for setters in ECL_SETTERS:
        apply_setters(E, setters)
        ref, st_ref = oracle_refs(case, models, setters)
        assert np.array_equal(st_ref, status)
        for m, o in enumerate(ref):
            ahead, st, b = E.run_build(models[m], True)
            instep, st2, b2 = E.run_build(models[m], False)
            assert st == st2 == o["status"]
            assert np.array_equal(ahead, instep), m
            if st:
                assert (ahead == -1.0).all()
            else:
                assert b == b2 == build
                assert relerr(ahead, o["spectrum"]) < 1e-9, m

