"""CPU: the transit tile kernels the built library holds, and their register fit.

Both transit kernels run 2 CTAs of 256 threads per SM (`__launch_bounds__(256, 2)`), which caps them
at 128 registers.  The specialised builds cover 1-4 grid molecules with 0-2 CIA files; every other
configuration takes the run-time-count build (0, -1).  The tensor-core (DMMA) kernel has a build with
and without the scattering / cloud terms; the DFMA tile kernel also serves the introspection
(`keep`) launches.  A stack frame or local memory would put spills on the shared-memory pipe that
both kernels are bound by.

The register ceilings are what each build uses with the CUDA 12.9 toolchain for sm_100a.  A build
that needs more has had its generated code changed; both kernels are sensitive to that (a rise of
two registers in one build came with a 0.7 % slower W12 launch in another), so a change to their
code has to be checked on the GPU before a ceiling is raised."""
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SPECIALISED = [(nmol, ncia) for nmol in range(1, 5) for ncia in range(3)] + [(0, -1)]

# (NMOL, NCIA) -> registers of transit_mma_kernel<NMOL, NCIA, false, SC> for SC false, true
MMA_REGS = {(0, -1): (127, 128),
            (4, 2): (121, 122), (4, 1): (104, 104), (4, 0): (96, 96),
            (3, 2): (121, 122), (3, 1): (96, 102), (3, 0): (94, 94),
            (2, 2): (112, 116), (2, 1): (94, 96), (2, 0): (94, 94),
            (1, 2): (96, 108), (1, 1): (94, 94), (1, 0): (94, 94)}
# transit_tile_kernel<NMOL, NCIA, KEEP>: 124 registers, except <4, 2, false>
TILE_REGS = {(4, 2, 0): 126}


def transit_usage():
    out = subprocess.run(["cuobjdump", "-res-usage", os.path.join(ROOT, "bart_b200", "libbart_b200.so")],
                         capture_output=True, text=True, check=True).stdout
    usage = {}
    for kern, args, regs, stack, local in re.findall(
            r"Function _ZN4bart\d+(transit_tile_kernel|transit_mma_kernel)I(\w+?)EEv\w*:\s*"
            r"REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out):
        targs = tuple(int(v.replace("n", "-")) for v in re.findall(r"L[ib](n?\d+)E", args))
        assert (kern, targs) not in usage, (kern, targs)
        usage[(kern, targs)] = (int(regs), int(stack), int(local))
    return usage


def test_transit_instantiations(built):
    u = transit_usage()
    tile = {a for k, a in u if k == "transit_tile_kernel"}
    mma = {a for k, a in u if k == "transit_mma_kernel"}
    # <NMOL, NCIA, KEEP>: the production builds, and the introspection build with run-time counts
    assert tile == {(n, c, 0) for n, c in SPECIALISED} | {(0, -1, 1)}, sorted(tile)
    # <NMOL, NCIA, KEEP, SC>: production only
    assert mma == {(n, c, 0, sc) for n, c in SPECIALISED for sc in (0, 1)}, sorted(mma)


def test_transit_builds_keep_their_register_fit(built):
    u = transit_usage()
    assert len(u) == 40
    for (kern, targs), (regs, stack, local) in u.items():
        if kern == "transit_mma_kernel":
            cap = MMA_REGS[targs[:2]][targs[3]]
        else:
            cap = TILE_REGS.get(targs, 124)
        assert regs <= cap and stack == 0 and local == 0, (kern, targs, regs, stack, local, cap)
