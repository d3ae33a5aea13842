"""ProbOhemCrossEntropy2d without a GPU: the C ABI's argument checks, the Python module's refusals, and the test-only
restatement oracle/ohem_ref.py against the reference's own class (loss.py:8-46) when a checkout of it is available."""
import ctypes
import importlib.util
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("CSS_REFERENCE_ROOT") or os.path.join(ROOT, "baseline", "_ref")
REF_LOSS = os.path.join(REF, "generalframeworks", "loss", "loss.py")


def test_ohem_abi_argument_errors_without_a_gpu():
    from css_b200 import _lib
    lib = _lib.load()
    one = ctypes.c_void_p(256)
    B, C, H, W = 2, 19, 33, 35
    nbytes = lib.css_ohem_workspace_bytes(B, H, W)
    assert nbytes >= 3 * 4 * B * H * W                        # p_t, lse, nll per pixel at least
    assert lib.css_ohem_workspace_bytes(0, H, W) == 0 and lib.css_ohem_workspace_bytes(B, -1, W) == 0
    assert lib.css_ohem_workspace_bytes(2 ** 15, 2 ** 9, 2 ** 8) == 0          # 2^32 pixels: beyond int32 pixel ids
    fwd = lib.css_ohem_forward
    # every call below fails its argument check before anything is launched
    args = [one, one, None, 255, 0.7, 256, B, C, H, W, one, nbytes, one, one, one, None]
    for i in (0, 1, 10, 12, 13, 14):                                          # every required pointer
        a = list(args)
        a[i] = None
        assert fwd(*a) == -1 and b"null" in lib.css_last_error()
    for i, v in ((6, 0), (7, 0), (8, -3), (9, 0), (6, 70000)):               # sizes
        a = list(args)
        a[i] = v
        assert fwd(*a) == -1, (i, v)
    a = list(args)
    a[11] = nbytes - 1
    assert fwd(*a) == -4 and b"workspace" in lib.css_last_error()
    a = list(args)
    a[6], a[8], a[9] = 2 ** 15, 2 ** 9, 2 ** 8
    assert fwd(*a) == -4
    bargs = [one, one, one, None, B, C, H, W, one, nbytes, one, None]
    for i in (0, 1, 2, 8, 10):
        b = list(bargs)
        b[i] = None
        assert lib.css_ohem_backward(*b) == -1
    b = list(bargs)
    b[9] = 16
    assert lib.css_ohem_backward(*b) == -4
    b = list(bargs)
    b[5] = 0
    assert lib.css_ohem_backward(*b) == -1
    with pytest.raises(RuntimeError, match="css_ohem_forward"):
        _lib.check(-1, "css_ohem_forward")


def test_ohem_module_refuses_cpu_tensors_and_other_reductions():
    import css_b200
    crit = css_b200.ProbOhemCrossEntropy2d(ignore_index=255, thresh=0.7, min_kept=100)
    with pytest.raises(RuntimeError, match="CUDA"):
        crit(torch.zeros(1, 19, 8, 8), torch.zeros(1, 8, 8, dtype=torch.long))
    with pytest.raises(ValueError, match="mean"):
        css_b200.ProbOhemCrossEntropy2d(ignore_index=255, reduction="sum")
    w = css_b200.ProbOhemCrossEntropy2d(ignore_index=255, use_weight=True, down_ratio=8)
    assert w.weight.shape == (19,) and w.down_ratio == 8 and w.thresh == 0.6 and w.min_kept == 256


def _reference_class():
    """The reference's own ProbOhemCrossEntropy2d, loaded from its file under a private module name (install() may already
    have replaced the name in generalframeworks.loss.loss)."""
    if REF not in sys.path:
        sys.path.insert(0, REF)
    spec = importlib.util.spec_from_file_location("_css_reference_loss_for_ohem", REF_LOSS)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.ProbOhemCrossEntropy2d


@pytest.mark.skipif(not os.path.isfile(REF_LOSS), reason="no reference checkout: set CSS_REFERENCE_ROOT or stage baseline/_ref")
@pytest.mark.parametrize("use_weight", [False, True])
def test_restatement_matches_the_reference_class(use_weight):
    from css_b200 import synth
    from oracle import ohem_ref
    Ref = _reference_class()
    B, C, H, W = 2, 19, 24, 28
    g = synth._gen(21)
    cls = synth.class_map(B, C, H, W, g, ignore_frac=0.1, block=4)
    target = torch.where(cls < 0, torch.full_like(cls, 255), cls)
    n_valid = int((target != 255).sum())
    untrained = synth.logits_for(cls, C, g)
    confident = 6.0 * torch.nn.functional.one_hot(cls.clamp_min(0), C).permute(0, 3, 1, 2).float() + torch.randn(B, C, H, W, generator=g)
    cases = [(untrained, 0.7, 200),                      # T = thresh
             (confident, 0.7, n_valid // 2),             # T = the min_kept-th smallest p_t
             (untrained, 0.7, n_valid + 1),              # no OHEM: plain CE over the valid pixels
             (untrained, 0.7, 0)]                        # min_kept = 0: plain CE
    for pred, thresh, min_kept in cases:
        kw = dict(ignore_index=255, thresh=thresh, min_kept=min_kept, use_weight=use_weight)
        p1 = pred.clone().requires_grad_(True)
        p2 = pred.clone().requires_grad_(True)
        l1 = Ref(**kw)(p1, target.clone())
        l2 = ohem_ref.ProbOhemCrossEntropy2d(**kw)(p2, target.clone())
        l1.backward()
        l2.backward()
        assert torch.equal(l1, l2), (min_kept, l1.item(), l2.item())
        assert torch.equal(p1.grad, p2.grad)


def test_ohem_kernels_keep_everything_in_registers():
    """No local-memory traffic (spills or stack arrays) in any of the OHEM kernels: the C logits of a pixel stay in registers."""
    import re
    import shutil
    import subprocess
    from css_b200 import build
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not available")
    sass = subprocess.run(["cuobjdump", "-sass", build.build()], capture_output=True, text=True).stdout
    funcs = re.findall(r"Function : (\S*ohem_\S*)\n(.*?)(?=Function : |\Z)", sass, flags=re.S)
    assert len(funcs) >= 14, "OHEM kernels not found"
    for name, body in funcs:
        assert not re.search(r"\b(LDL|STL)\b", body), f"{name}: local-memory access"


@pytest.mark.skipif(not os.path.isfile(REF_LOSS), reason="no reference checkout: set CSS_REFERENCE_ROOT or stage baseline/_ref")
def test_install_patches_the_ohem_loss():
    import css_b200
    from css_b200 import install, models
    saved_hooks = dict(vars(models.hooks))
    try:
        _, ref_loss = install.install(reference_root=REF)
        assert ref_loss.ProbOhemCrossEntropy2d is css_b200.ProbOhemCrossEntropy2d
        crit = ref_loss.ProbOhemCrossEntropy2d(ignore_index=255, thresh=0.7, min_kept=200000, use_weight=False)
        assert (crit.ignore_index, crit.thresh, crit.min_kept) == (255, 0.7, 200000)
    finally:
        for k, v in saved_hooks.items():
            setattr(models.hooks, k, v)
