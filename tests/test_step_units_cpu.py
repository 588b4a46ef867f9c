"""CPU: every step kernel sits in a translation unit of its own (DESIGN.md section 7).  With two step kernels in one unit
ptxas shares the out-of-line device functions between them, and the staged kernel once lost a third of its speed that
way.  Read from `cuobjdump -res-usage` of the built library, which lists each unit's functions under
`identifier = <unit>`."""
import functools
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "openkitchen_b200", "lib", "libopenkitchen_b200.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"

# mangled name -> (unit, stack frame limit in bytes).  The limits are the stack frames the kernels are built with (CUDA
# 12.9): a kernel change that moves them is to update them on purpose.  The last template argument is the StepVariant:
# 0 plain, 1 drawn, 2 laps.
EXPECTED = {
    "_ZN2ok16beam_step_kernelILb1ELb0ELNS_11StepVariantE0EEEvNS_10StepParamsENS_8ActorArgIXT0_EE4typeE": ("ok_step_staged.cu", 56),
    "_ZN2ok16beam_step_kernelILb0ELb0ELNS_11StepVariantE0EEEvNS_10StepParamsENS_8ActorArgIXT0_EE4typeE": ("ok_step_unstaged.cu", 56),
    "_ZN2ok16beam_step_kernelILb0ELb1ELNS_11StepVariantE0EEEvNS_10StepParamsENS_8ActorArgIXT0_EE4typeE": ("ok_step_actor.cu", 80),
    "_ZN2ok16grid_step_kernelILNS_11StepVariantE0EEEvNS_10StepParamsE": ("ok_step_grid.cu", 0),
    "_ZN2ok16beam_step_kernelILb1ELb0ELNS_11StepVariantE1EEEvNS_10StepParamsENS_8ActorArgIXT0_EE4typeE": ("ok_step_staged_drawn.cu", 56),
    "_ZN2ok16beam_step_kernelILb0ELb0ELNS_11StepVariantE1EEEvNS_10StepParamsENS_8ActorArgIXT0_EE4typeE": ("ok_step_unstaged_drawn.cu", 56),
    "_ZN2ok16beam_step_kernelILb0ELb1ELNS_11StepVariantE1EEEvNS_10StepParamsENS_8ActorArgIXT0_EE4typeE": ("ok_step_actor_drawn.cu", 80),
    "_ZN2ok16grid_step_kernelILNS_11StepVariantE1EEEvNS_10StepParamsE": ("ok_step_grid_drawn.cu", 0),
    "_ZN2ok16beam_step_kernelILb1ELb0ELNS_11StepVariantE2EEEvNS_10StepParamsENS_8ActorArgIXT0_EE4typeE": ("ok_step_staged_laps.cu", 136),
    "_ZN2ok16beam_step_kernelILb0ELb0ELNS_11StepVariantE2EEEvNS_10StepParamsENS_8ActorArgIXT0_EE4typeE": ("ok_step_unstaged_laps.cu", 120),
    "_ZN2ok16beam_step_kernelILb0ELb1ELNS_11StepVariantE2EEEvNS_10StepParamsENS_8ActorArgIXT0_EE4typeE": ("ok_step_actor_laps.cu", 160),
    "_ZN2ok16grid_step_kernelILNS_11StepVariantE2EEEvNS_10StepParamsE": ("ok_step_grid_laps.cu", 40),
}
# demangled: ok::beam_step_kernel<...> and ok::grid_step_kernel<...>, every __global__ step kernel
STEP_KERNEL_PREFIXES = ("_ZN2ok16beam_step_kernelI", "_ZN2ok16grid_step_kernelI")


@functools.cache
def _step_kernels():
    """{unit: {function: (registers, stack bytes)}} of every step kernel"""
    if not os.path.exists(CUOBJDUMP):
        pytest.skip("cuobjdump not found")
    if not os.path.exists(LIB):
        pytest.skip(f"{LIB} not built")
    out = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    units, unit, fn = {}, None, None
    for line in out.splitlines():
        if m := re.match(r"identifier = (.*)$", line.strip()):
            unit = m.group(1).strip()
        elif m := re.match(r"Function (\S+):$", line.strip()):
            fn = m.group(1)
        elif fn and (m := re.search(r"REG:(\d+) STACK:(\d+)", line)):
            if fn.startswith(STEP_KERNEL_PREFIXES):
                units.setdefault(unit, {})[fn] = (int(m.group(1)), int(m.group(2)))
            fn = None
    return units


def test_one_step_kernel_per_unit():
    units = _step_kernels()
    for unit, fns in units.items():
        assert len(fns) == 1, f"{unit} holds {len(fns)} step kernels: {sorted(fns)}"
    found = {fn: unit for unit, fns in units.items() for fn in fns}
    assert found == {fn: unit for fn, (unit, _) in EXPECTED.items()}


def test_step_kernels_keep_their_registers_and_stack():
    units = _step_kernels()
    for fn, (unit, stack_limit) in EXPECTED.items():
        regs, stack = units[unit][fn]
        assert regs <= 64, f"{unit}: {regs} registers"
        assert stack <= stack_limit, f"{unit}: {stack}-byte stack frame, was {stack_limit}"
