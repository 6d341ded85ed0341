"""The occupancy DESIGN.md claims for the heavy kernels, checked on the built library (cuobjdump -res-usage, no GPU needed):
registers per thread at or under the cap that lets the stated number of CTAs share an SM's 64 K registers.  (Shared memory
is dynamic; its budgets are static_asserts beside the work structs in idocp_b200/csrc.)"""
import re
import shutil
import subprocess

import pytest

import __graft_entry__ as g

# kernel name fragment -> (threads per CTA, CTAs per SM)
BUDGET = {
    "k_fb_riccati_backward": (128, 4),
    "k_fb_condense": (128, 6),
    "k_fb_robotILb0": (192, 2),
    "k_fb_robotILb1": (192, 2),
    "k_fb_update": (64, 16),
    "k_parnmpc_invert": (128, 4),
    "k_update_linearizeILb0ELb0": (128, 2),
    "k_riccatiILb0": (128, 2),
}


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not installed")
def test_register_budgets_of_the_heavy_kernels():
    lib = g.build_cuda()
    out = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True, check=True).stdout
    regs = {}
    for name, r in re.findall(r"Function (\S+):\s*\n\s*REG:(\d+)", out):
        regs[name] = int(r)
    assert regs, "no kernels found in the library"
    for frag, (threads, ctas) in BUDGET.items():
        hits = {n: r for n, r in regs.items() if frag in n}
        assert hits, frag
        for n, r in hits.items():
            alloc = -(-r // 8) * 8                     # registers are allocated in units of 8 per thread
            assert alloc * threads * ctas <= 65536, (n, r, threads, ctas)


NO_SPILLS = ["k_parnmpc_invert", "k_fb_riccati_backward", "k_fb_condense", "k_update_linearizeILb0ELb0", "k_fb_expand", "k_expandILb0ELb0ELb0"]


def test_kernels_documented_as_spill_free_have_no_spills():
    """ptxas -v of the product build (build_ptxas.log, written by __graft_entry__.build_cuda): the kernels DESIGN.md calls
    spill-free report 0 bytes of spill stores / loads."""
    import os
    g.build_cuda(force=not os.path.exists(os.path.join(g.ROOT, "build_ptxas.log")))
    log = open(os.path.join(g.ROOT, "build_ptxas.log")).read()
    blocks = re.findall(r"Function properties for (\S+)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", log)
    assert blocks
    for frag in NO_SPILLS:
        hits = [(n, int(st), int(ld)) for n, _, st, ld in blocks if frag in n]
        assert hits, frag
        for n, st, ld in hits:
            assert st == 0 and ld == 0, (n, st, ld)


# the only macros a preprocessor conditional in idocp_b200/csrc may test, besides include guards: the SIMT-emulator build
# and the storage class of the generated ANYmal tables
ALLOWED_CONDITIONS = {"IDOCP_B200_EMU", "ANYMAL_TABLE"}


def test_kernel_sources_compile_one_way():
    """The launch bounds, prefetches and code paths the benchmarks measure are the only ones in the sources: no `-D` flag can
    select another variant of a kernel.  Every #if / #ifdef / #ifndef / #elif tests IDOCP_B200_EMU or ANYMAL_TABLE, or is an
    include guard (#ifndef X directly followed by a bare #define X)."""
    import os
    csrc = os.path.join(g.ROOT, "idocp_b200", "csrc")
    bad = []
    for f in sorted(os.listdir(csrc)):
        lines = open(os.path.join(csrc, f)).read().splitlines()
        for i, line in enumerate(lines):
            m = re.match(r"\s*#\s*(if|ifdef|ifndef|elif)\b(.*)", line)
            if not m:
                continue
            cond = re.sub(r"//.*|/\*.*?\*/", "", m.group(2))
            names = set(re.findall(r"[A-Za-z_]\w*", cond)) - {"defined"}
            nxt = next((l.strip() for l in lines[i + 1:] if l.strip()), "")
            if m.group(1) == "ifndef" and len(names) == 1 and nxt == "#define " + next(iter(names)):
                continue
            if not names or not names <= ALLOWED_CONDITIONS:
                bad.append("%s:%d: %s" % (f, i + 1, line.strip()))
    assert not bad, "build switches in the kernel sources:\n" + "\n".join(bad)
