"""Register and shared-memory footprint of the resident kernel's default launch shape (DESIGN.md 4.1).  CPU only.

C1 runs four co-resident problems per launch, four 4-warp CTAs on every SM, in one of the two 128-register instantiations
(k_resident_t<160, 3> or <128, 4>; the host takes the first in its list that fits).  The 128-register budget holds the
PCG state only while nothing of it goes to local memory inside the PCG loop: at four CTAs the shared-memory carve-out
leaves so little L1 that spill reloads come from L2, in a loop that is already latency-bound.  And the strip arrays of
four CTAs have to fit one SM's shared memory, or the host falls back to three problems per launch.

solver_resident.cu is compiled for sm_100a with the Makefile's flags (which include -Xptxas -v), inside a translation
unit that adds one probe kernel whose static shared memory is exactly one StripSmem, so that ptxas reports its size."""
import os
import re
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "arap_flow_b200", "csrc")
SRC = os.path.join(CSRC, "solver_resident.cu")

KERNELS = ["k_resident_tILi128ELi4ELb0EE", "k_resident_tILi160ELi3ELb0EE"]  # k_resident_t<128, 4> and <160, 3>
CTAS, WARPS = 4, 4                        # per SM, per CTA
SM_SHARED = 228 * 1024                    # shared memory of one sm_100 SM
CTA_RESERVED = 1024                       # the driver's reservation per resident CTA

PROBE = r"""
#include "%s"
namespace arapb200 {
__global__ void k_footprint_probe(int* out)
{
    __shared__ StripSmem strip;
    out[threadIdx.x] = reinterpret_cast<volatile int*>(&strip)[threadIdx.x];
}
}
"""


def _tools():
    nvflags = subprocess.run(["make", "-s", "--no-print-directory", "-C", CSRC, "--eval",
                              "print-nvflags: ; @echo $(NVCC) $(NVFLAGS)", "print-nvflags"],
                             capture_output=True, text=True, check=True).stdout.split()
    nvcc = nvflags[0]
    bindir = os.path.dirname(nvcc)
    tools = [nvcc] + [os.path.join(bindir, t) for t in ("cuobjdump", "nvdisasm")]
    for t in tools:
        if not (os.path.isfile(t) or shutil.which(t)):
            pytest.skip(f"{t} not available")
    return nvflags, tools[1], tools[2]


@pytest.fixture(scope="module")
def build(tmp_path_factory):
    nvflags, cuobjdump, nvdisasm = _tools()
    assert "-Xptxas" in nvflags and "-v" in nvflags
    d = tmp_path_factory.mktemp("footprint")
    probe = d / "probe.cu"
    probe.write_text(PROBE % SRC)
    r = subprocess.run(nvflags + ["-I", CSRC, "-c", "-o", str(d / "probe.o"), str(probe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    subprocess.run([cuobjdump, "-xelf", "all", "probe.o"], cwd=d, capture_output=True, check=True)
    cubins = [f for f in os.listdir(d) if f.endswith(".cubin")]
    assert len(cubins) == 1, cubins
    sass = subprocess.run([nvdisasm, "-gi", "-c", str(d / cubins[0])], capture_output=True, text=True,
                          check=True).stdout
    return r.stderr, sass


def _ptxas(log, pattern):
    """(stack, spill stores, spill loads, registers, static smem) of the one entry function matching pattern"""
    blocks = re.split(r"ptxas info\s*: Compiling entry function", log)
    hits = [b for b in blocks if re.search(pattern, b.splitlines()[0])]
    assert len(hits) == 1, (pattern, len(hits))
    b = hits[0]
    m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", b)
    u = re.search(r"Used (\d+) registers.*?(\d+) bytes smem", b)
    assert m and u, b
    return tuple(int(x) for x in m.groups()) + (int(u.group(1)), int(u.group(2)))


def _pcg_loop_lines():
    """first and last source line of the PCG iteration loop in solver_resident.cu"""
    lines = open(SRC, encoding="utf-8").read().splitlines()
    first = [i + 1 for i, l in enumerate(lines) if "for (int it = 0; it < P.nPCG; ++it) {" in l]
    assert len(first) == 1, first
    indent = lines[first[0] - 1].index("for")
    last = next(i + 1 for i in range(first[0], len(lines)) if lines[i].startswith(" " * indent + "}"))
    return first[0], last


def _local_accesses(sass, kernel):
    """(source line in solver_resident.cu, mnemonic) of every LDL / STL of the kernel"""
    out, inside, line = [], False, None
    for l in sass.splitlines():
        m = re.match(r"\s*\.text\.(\S+):", l)
        if m:
            inside = kernel in m.group(1)
            continue
        if not inside:
            continue
        m = re.search(r'//## File "([^"]+)", line (\d+)', l)
        if m:
            line = int(m.group(2)) if os.path.basename(m.group(1)) == "solver_resident.cu" else None
            continue
        m = re.search(r"\b(LDL|STL)\b", l)
        if m:
            out.append((line, m.group(1)))
    return out


@pytest.mark.parametrize("kernel", KERNELS)
def test_128_register_kernels_keep_the_pcg_loop_out_of_local_memory(build, kernel):
    log, sass = build
    stack, st, ld, regs, _ = _ptxas(log, kernel)
    assert regs <= 128
    acc = _local_accesses(sass, kernel)
    first, last = _pcg_loop_lines()
    in_loop = [a for a in acc if a[0] is not None and first <= a[0] <= last]
    # what is left in the loop's lines is one reload per iteration (the trace write's thread predicate, behind the second
    # barrier) and one on the loop's exit; with q in registers and the masks hoisted out of the loop it was 52 (288 B of stack)
    assert len(in_loop) <= 2, (in_loop, (first, last), (stack, st, ld))
    assert stack <= 64, (stack, st, ld)


@pytest.mark.parametrize("kernel", KERNELS)
def test_four_ctas_of_four_strips_fit_one_sm(build, kernel):
    log, _ = build
    strip = _ptxas(log, "k_footprint_probe")[4]
    static = _ptxas(log, kernel)[4]
    per_cta = WARPS * strip + static + CTA_RESERVED
    assert CTAS * per_cta <= SM_SHARED, (strip, static, CTAS * per_cta)
