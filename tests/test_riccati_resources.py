"""k_riccati, the serial backward Riccati sweep of UnOCPSolver, holds a whole stage in registers and per-octet tiles: ptxas -v
of the product build reports no stack frame and no spill stores or loads for either instantiation, and few enough registers
for two CTAs of RIC_THREADS per SM.  A spill there sits on the sweep's dependent chain 20 times per instance group."""
import os
import re

import __graft_entry__ as g


def test_riccati_sweep_is_spill_free():
    g.build_cuda(force=not os.path.exists(os.path.join(g.ROOT, "build_ptxas.log")))
    log = open(os.path.join(g.ROOT, "build_ptxas.log")).read()
    blocks = re.findall(r"Function properties for (\S*k_riccati\S*)\n\s*(\d+) bytes stack frame, (\d+) bytes spill stores, "
                        r"(\d+) bytes spill loads\n[^\n]*Used (\d+) registers", log)
    assert len(blocks) == 2, blocks
    for name, stack, st, ld, regs in blocks:
        assert (int(stack), int(st), int(ld)) == (0, 0, 0), (name, stack, st, ld)
        assert -(-int(regs) // 8) * 8 * 128 * 2 <= 65536, (name, regs)
