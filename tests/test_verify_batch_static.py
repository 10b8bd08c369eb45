"""Static checks of the batch verifier's kernels inside the built library (CPU; cuobjdump ships with the CUDA toolkit): all four are
present and keep their state in registers — no stack frame, no local memory (the Keccak path walks and the AIR folding at zeta
would otherwise spill per-thread arrays)."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "valida_b200", "libvalida_b200.so")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"

pytestmark = pytest.mark.skipif(not (os.path.exists(LIB) and os.path.exists(CUOBJDUMP)), reason="needs the built library and cuobjdump")


def test_batch_verifier_kernels_present_without_stack_or_local_memory():
    out = subprocess.run([CUOBJDUMP, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    res = {m.group(1): (int(m.group(2)), int(m.group(3)), int(m.group(4)))
           for m in re.finditer(r"Function (\S+):\s*\n\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out)}
    for name, count in (("verify_merkle_kernel", 1), ("verify_open_kernel", 1), ("verify_fold_kernel", 1), ("verify_constraints_kernel", 14)):
        found = {k: v for k, v in res.items() if name in k}
        assert len(found) == count, (name, sorted(found))
        for k, (reg, stack, local) in found.items():
            assert stack == 0 and local == 0, (k, reg, stack, local)
