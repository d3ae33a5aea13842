"""CPU guard on the machine code of the fp32 gradient scorer (score_ce_kernel<true, false, true, FIX, float>, whole-warp rows):
no local-memory traffic, and the 16 128-bit loads of a batch (8 rows x 2 LDG.128 per lane) issued back to back -- only the
shuffles that hand out the row ids may sit between them, no FFMA2 and no reduction -- so a warp has all 8 rows in flight at
once.  A schedule that splits them pays the L2 round trip more than once per batch."""
import re
import shutil
import subprocess

import pytest


def test_fp32_gradient_scorer_sass():
    from css_b200 import build
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not available")
    sass = subprocess.run(["cuobjdump", "-sass", build.build()], capture_output=True, text=True, check=True).stdout
    funcs = re.findall(r"Function : (\S*score_ce_kernelILb1ELb0ELb1ELb[01]EfE\S*)\n(.*?)(?=Function : |\Z)", sass, flags=re.S)
    assert len(funcs) == 2, f"expected the two fp32 gradient instantiations, found {[n for n, _ in funcs]}"
    for name, body in funcs:
        ops = re.findall(r"^\s+/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", body, flags=re.M)
        local = [op for op in ops if op.startswith(("LDL", "STL"))]
        assert not local, f"{name}: local-memory traffic {local[:4]}"
        best = run = 0
        for op in ops:
            if op.startswith("LDG.E.128"):
                run += 1
                best = max(best, run)
            elif op.startswith(("FFMA2", "FMUL2", "SHFL.BFLY", "LDS")):
                run = 0
        assert best >= 16, f"{name}: row loads split by compute (longest run of LDG.E.128 = {best})"
