"""Register / spill budgets of the three hot kernels, read from the ptxas logs the build writes (csrc/*.ptxas.log).

The numbers are the ones DESIGN.md quotes: k_extend / k_shadow at 64 registers (8 blocks of 128 threads per SM),
k_shade at 128 registers WITHOUT spills in the reference mode (the register diet: the hit geometry is reduced to its
results before the material fetch), at 128 registers with its spills reported in the emissive-MIS mode.  A change that
brings the spills back shows up here, on the CPU, before any GPU time is spent."""
import os
import re

import pytest

import conftest

LOG = os.path.join(conftest.ROOT, "path-tracing_b200", "csrc", "wavefront.ptxas.log")


def kernel_stats():
    """{(kernel, ALPHA, STATS, EMISSIVE): (registers, spill store bytes, spill load bytes, stack bytes)} of wavefront.cu;
    EMISSIVE is k_shade's third template flag, False for k_extend and k_shadow."""
    if not os.path.exists(LOG):
        import importlib

        importlib.import_module("path-tracing_b200.core").build()
    text = open(LOG).read()
    out = {}
    for m in re.finditer(r"Function properties for (\S+)\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n"
                         r"ptxas info\s+: Used (\d+) registers", text):
        name = m[1]
        k = re.search(r"(k_extend|k_shade|k_shadow)ILb([01])ELb([01])E(?:Lb([01])E)?", name)
        if k:
            out[(k[1], int(k[2]), int(k[3]), k[4] == "1")] = (int(m[5]), int(m[3]), int(m[4]), int(m[2]))
    return out


def test_hot_kernels_keep_their_register_budgets_per_shade_mode():
    st = kernel_stats()
    assert len(st) == 16, sorted(st)  # (k_extend, k_shadow) x (ALPHA, STATS) + k_shade x (ALPHA, STATS, EMISSIVE)
    for (kernel, alpha, stats, emissive), (regs, spill_st, spill_ld, stack) in st.items():
        if kernel == "k_shade":
            assert regs <= 128, (kernel, alpha, stats, emissive, regs)
            if not stats and not emissive:
                assert spill_st == 0 and spill_ld == 0, (kernel, alpha, stats, emissive, spill_st, spill_ld)
        else:
            assert not emissive, (kernel, alpha, stats)
            assert regs <= 64, (kernel, alpha, stats, regs)  # 8 blocks x 128 threads resident per SM
            # the traversal stack (96 entries x 8 B) lives in local memory by design; everything else is the spill frame
            assert stack <= 96 * 8 + 256, (kernel, alpha, stats, stack)


def test_emissive_k_shade_register_budget():
    """k_shade<*, *, true>: 128 registers at most, like the reference mode (four 128-thread blocks per SM); its spills
    are reported."""
    found = 0
    for (kernel, alpha, stats, emissive), (regs, spill_st, spill_ld, _) in sorted(kernel_stats().items()):
        if kernel == "k_shade" and emissive:
            found += 1
            print(f"k_shade<{alpha},{stats},true>: {regs} registers, spills {spill_st} / {spill_ld} bytes (stores / loads)")
            assert regs <= 128, (alpha, stats, regs)
    assert found == 4
