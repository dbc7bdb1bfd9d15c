"""CPU: the register budget of the eclipse throughput kernel, read from the built library.

Batches beyond one resident wave take the form that runs 10 CTAs of 64 threads (20 warps) per SM
for the specialised builds with at most one CIA file, which caps it at 96 registers; its time per
launch depends on that occupancy and on not spilling (local memory goes through the L1 data pipe,
the kernel's busiest unit).  The
builds with two CIA files, the run-time-count build and the introspection build keep 8 CTAs
(128 registers) and must not spill either."""
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def eclipse_column_usage():
    out = subprocess.run(["cuobjdump", "-res-usage", os.path.join(ROOT, "bart_b200", "libbart_b200.so")],
                         capture_output=True, text=True, check=True).stdout
    usage = {}
    for name, regs, stack, local in re.findall(
            r"Function (_ZN4bart21eclipse_column_kernelI\w+):\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out):
        m = re.match(r"_ZN4bart21eclipse_column_kernelILi(\d+)ELi(n?\d+)ELi(\d+)ELb([01])ELi(n?\d+)ELb([01])ELb([01])E", name)
        nmol, ncia, nang, keep, sq, sc, ahead = (int(g.replace("n", "-")) for g in m.groups())
        if not ahead:                 # the form that loads one depth ahead serves small batches only
            usage[(nmol, ncia, nang, keep, sq, sc)] = (int(regs), int(stack), int(local))
    return usage


def test_bench_instantiation_fits_96_registers_without_spilling(built):
    u = eclipse_column_usage()
    # W12: 4 molecules, 1 CIA file, the default 5-angle ray grid (angle 3 = angle 0 squared), no
    # scattering / cloud terms
    regs, stack, local = u[(4, 1, 5, 0, 0x03, 0)]
    assert regs <= 96 and stack == 0 and local == 0, (regs, stack, local)


def test_eclipse_builds_do_not_spill(built):
    u = eclipse_column_usage()
    assert len(u) == 50, sorted(u)
    # every build except the run-time angle count with 4 molecules and one CIA file, which spilled
    # more than this at 128 registers as well
    spilling = {k for k, (r, s, l) in u.items() if s or l}
    assert spilling <= {(4, 1, 0, 0, -1, 0), (4, 1, 0, 0, -1, 1)}, sorted(spilling)
    for (nmol, ncia, nang, keep, sq, sc), (regs, _, _) in u.items():
        cap = 96 if 1 <= nmol <= 4 and 0 <= ncia <= 1 and not keep else 128
        assert regs <= cap, ((nmol, ncia, nang, keep, sq, sc), regs)
