"""Valid-list entries {pixel id, bits of 1 / max(||r||, 1e-8)}: what css_select_lists writes and what every scorer reads.

  * The entries' ids are the row-major valid pixels of each class (the hard list likewise), and their inverse norms are
    bitwise torch's 1 / clamp_min(norms, 1e-8) of the norms the scorer is handed: fp32, bf16 and channels-last maps.
  * A rows cache checked against DistributedDataParallel's clone of a changed map ("verify"): the flag is raised, the norms
    are refreshed, and the entries carry the refreshed norms, so the loss equals the plain "miss" run's bit for bit.
  * Every scorer form on fed draws gives the bits recorded in tests/golden/scorer_fed_bits.json (written by the build that
    still loaded each candidate's norm and divided in the scorer: `python -m tests.test_gpu_list_entries --write`).
"""
import hashlib
import json
import os
import sys

import pytest
import torch

from tests import test_gpu_kernel_matrix as M

pytestmark = pytest.mark.gpu
lib = M.lib
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "scorer_fed_bits.json")


def check_entries(crit, rep, label, mask, prob, strong):
    from css_b200 import _lib
    ws, norms = crit.last["ws"], crit.last["norms"]
    B2, C, h, w = label.shape
    N = ws.N
    meta = ws.meta.cpu()
    entries = ws.valid_list.view(C, N, 2).cpu()
    hard = ws.hard_list.view(C, N).cpu()
    valid = (label * mask).permute(1, 0, 2, 3).reshape(C, N) != 0            # css_select: label * mask != 0 (loss.py:80)
    is_hard = valid & (prob.permute(1, 0, 2, 3).reshape(C, N) < strong)
    inv_bits = (1.0 / norms.clamp_min(1e-8)).view(torch.int32).cpu()
    seen = 0
    for c in range(C):
        ids = torch.nonzero(valid[c]).flatten().to(torch.int32).cpu()
        nv, nh = int(meta[_lib.META_N_VALID + c]), int(meta[_lib.META_N_HARD + c])
        assert nv == ids.numel()
        assert torch.equal(entries[c, :nv, 0], ids)
        assert torch.equal(entries[c, :nv, 1], inv_bits[ids.long()])
        assert torch.equal(hard[c, :nh], torch.nonzero(is_hard[c]).flatten().to(torch.int32).cpu())
        seen += nv
    assert seen > 0


def used_entries(crit):
    """The written prefix of every class's valid list (the rest of the buffer is never initialised)."""
    from css_b200 import _lib
    ws = crit.last["ws"]
    C, N = ws.key[1], ws.N
    meta = ws.meta.cpu()
    entries = ws.valid_list.view(C, N, 2).cpu()
    return [entries[c, :int(meta[_lib.META_N_VALID + c])].tolist() for c in range(C)]


@pytest.mark.parametrize("layout", ["fp32", "bf16", "channels_last"])
def test_entries(lib, layout):
    import css_b200
    B2, C, h, w, seed = 2, 7, 19, 23, 41
    rep, label, mask, prob, protos = M.scorer_inputs(B2, C, h, w, seed, torch.bfloat16 if layout == "bf16" else torch.float32)
    if layout == "channels_last":
        rep = M.to_channels_last(rep)
    rep[0, :, 0, 0] = 0                                            # a zero-norm valid pixel: its entry carries 1e8
    label[0, :, 0, 0] = 0
    label[0, 2, 0, 0] = 1
    mask[0, 0, 0, 0] = 1
    crit = css_b200.Contrast_Loss(num_queries=12, num_negatives=100, temp=0.5, strong_threshold=0.97, seed=seed).cuda()
    with torch.no_grad():
        crit(rep, label, mask, prob, protos.clone())
    assert crit.last["norms"][0].item() == 0
    check_entries(crit, rep, label, mask, prob, 0.97)


@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
def test_verify_clone_carries_refreshed_norms(lib, layout):
    """The cached rows and norms belong to `rep`; the loss gets a changed map at another address (version 0, as DDP's clone)."""
    import css_b200
    from css_b200 import _lib
    B2, C, h, w, seed = 2, 7, 24, 20, 2
    rep, label, mask, _, protos = M.scorer_inputs(B2, C, h, w, seed)
    if layout == "channels_last":
        rep = M.to_channels_last(rep)
    other = rep * 1.5 + 0.25
    other = M.to_channels_last(other) if layout == "channels_last" else other.contiguous()
    kw = dict(num_queries=8, num_negatives=64, temp=0.5, strong_threshold=0.8, seed=4)

    def run(rep_in, prob):
        crit = css_b200.Contrast_Loss(**kw).cuda()
        r = rep_in.detach().requires_grad_(True)
        loss = crit(r, label, mask, prob, protos.clone())
        loss.backward()
        return loss, r.grad, crit

    prob = css_b200.ops.proto_softmax_sim(rep, protos, 0.5)
    stale = prob._css_rows.norms.clone()
    loss, grad, crit = run(other, prob)
    assert crit.last["rows_cache_mode"] == "verify"
    assert int(crit.last["ws"].meta[_lib.META_ROWS_STALE].item()) == 1
    assert not torch.equal(crit.last["norms"], stale)
    check_entries(crit, other, label, mask, prob, 0.8)
    loss_ref, grad_ref, crit_ref = run(other, prob.clone())          # prob.clone() carries no rows: the plain pass
    assert crit_ref.last["rows_cache_mode"] == "miss"
    assert torch.equal(crit.last["norms"], crit_ref.last["norms"])
    assert used_entries(crit) == used_entries(crit_ref)
    assert loss.item() == loss_ref.item()
    assert torch.equal(grad, grad_ref)


FED_VARIANTS = ("grad-f32-reg", "grad-f32-ring", "grad-f32-bulk", "grad-bf16", "nograd-f32", "nograd-bf16")
FED_TEMPS = (0.5, 0.02)                                            # fixed-reference and online-max softmax


def _digest(*tensors):
    h = hashlib.sha256()
    for t in tensors:
        h.update(t.detach().reshape(-1).contiguous().view(torch.uint8).cpu().numpy().tobytes())
    return h.hexdigest()


def fed_bits(lib, variant, temp):
    """Loss, anchor pixels, updated prototypes and d loss / d anchor of one Contrast_Loss call on materialised draws, as a digest
    (the dense gradient is left out: grad_slab_kernel adds a pixel drawn as anchor three times or more in no fixed order)."""
    B2, C, h, w, Q, Nn, seed = 2, 7, 19, 23, 12, 100, 77
    dt = torch.bfloat16 if "bf16" in variant else torch.float32
    rep, label, mask, prob, protos = M.scorer_inputs(B2, C, h, w, seed, dt)
    kw = dict(num_queries=Q, num_negatives=Nn, temp=temp, strong_threshold=0.97, alpha=0.99)
    _, _, crit, _, _ = M.run_loss(lib, variant, rep, label, mask, prob, protos, kw, seed)
    a, n = crit.sample_indices(seed, 0)
    loss, grad, crit, _, p = M.run_loss(lib, variant, rep, label, mask, prob, protos, kw, seed, indices=(a, n))
    torch.cuda.synchronize()
    parts = [loss, crit.last["anchor_px"], p] + ([crit.last["grad_anchor"]] if grad is not None else [])
    return _digest(*parts)


@pytest.mark.parametrize("variant", FED_VARIANTS)
@pytest.mark.parametrize("temp", FED_TEMPS)
def test_fed_draws_bits_unchanged(lib, variant, temp):
    with open(GOLDEN) as f:
        golden = json.load(f)
    assert fed_bits(lib, variant, temp) == golden[f"{variant}@{temp}"]


if __name__ == "__main__":
    from css_b200 import _lib
    lib_ = _lib.load()
    lib_.css_set_rep_pass_path(0)
    out = {f"{v}@{t}": fed_bits(lib_, v, t) for v in FED_VARIANTS for t in FED_TEMPS}
    lib_.css_set_scorer_path(-1)
    text = json.dumps(out, indent=1, sort_keys=True) + "\n"
    if "--write" in sys.argv:
        with open(GOLDEN, "w") as f:
            f.write(text)
    print(text)
