"""CPU guard on the machine code of the fp32 gradient scorer (score_ce_kernel<true, false, true, FIX, float>, whole-warp rows):
a candidate's pixel id and inverse norm arrive together as one 8-byte valid-list entry, so the loops that gather the rows load
no norm and divide nothing.  The loops are found from their backward branches; the ones that hold one batch of row loads (16
LDG.E.128 per lane) are the batch loop and the loop over 32-id groups around it.  Inside them:
  * no MUFU.RCP and no CALL (the IEEE reciprocal 1 / max(||r||, 1e-8) is a MUFU.RCP with a called slow path);
  * the batch loop makes no 32-bit global load (it used to fetch the next group's norms);
  * the group loop fetches the entries as LDG.E.64, and at most one 32-bit global load is left (the fed negative index)."""
import re
import shutil
import subprocess

import pytest


def loops_with_one_batch(body):
    ins = [(int(a, 16), t.strip()) for a, t in re.findall(r"^\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", body, flags=re.M)]
    out = []
    for addr, text in ins:
        m = re.search(r"\bBRA\b.*?(0x[0-9a-f]+)", text)
        if m and int(m.group(1), 16) < addr:
            ops = [t for a, t in ins if int(m.group(1), 16) <= a <= addr]
            if sum("LDG.E.128" in o for o in ops) == 16:
                out.append(ops)
    return sorted(out, key=len)


def global_loads(ops, width):
    kinds = [re.search(r"\bLDG\.E(\.\d+)?", o) for o in ops]
    return sum(1 for k in kinds if k and (k.group(1) or "") == width)


def test_fp32_gradient_scorer_loads_entries():
    from css_b200 import build
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not available")
    sass = subprocess.run(["cuobjdump", "-sass", build.build()], capture_output=True, text=True, check=True).stdout
    funcs = re.findall(r"Function : (\S*score_ce_kernelILb1ELb0ELb1ELb[01]EfE\S*)\n(.*?)(?=Function : |\Z)", sass, flags=re.S)
    assert len(funcs) == 2, f"expected the two fp32 gradient instantiations, found {[n for n, _ in funcs]}"
    for name, body in funcs:
        loops = loops_with_one_batch(body)
        assert len(loops) >= 2, f"{name}: expected the batch loop and the id-group loop, found {len(loops)} loops with 16 row loads"
        for ops in loops:
            assert not any("MUFU.RCP" in o for o in ops), f"{name}: a reciprocal in the row loop"
            assert not any(re.search(r"\bCALL\b", o) for o in ops), f"{name}: a call (division slow path) in the row loop"
        batch, group = loops[0], loops[-1]
        assert global_loads(batch, "") == 0, f"{name}: 32-bit global loads in the batch loop"
        assert global_loads(group, ".64") >= 1, f"{name}: no 8-byte entry load in the id-group loop"
        assert global_loads(group, "") <= 1, f"{name}: {global_loads(group, '')} 32-bit global loads in the id-group loop"
