"""GPU parity of the fused ProbOhemCrossEntropy2d (DESIGN.md f-5) against oracle/ohem_ref.py, the statement-by-statement
restatement of the reference (loss.py:8-46), run on the same CUDA tensors.

Pass criteria everywhere: the kept mask, the threshold and the kept count are identical; loss within rel 1e-4; gradient within
rel 1e-4 with an identical zero pattern.  p_t is expected to be bit-identical to F.softmax (same serial class-order sum and the
same exp(x - max) / sum epilogue); the full-size tests print the largest ulp difference over the valid pixels and require 0."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ohem_ref

pytestmark = pytest.mark.gpu

CITY = dict(B=4, C=19, H=769, W=769)


def _confident(cls, C, g, margin=6.0, noise=1.0):
    """Logits of a trained network: the labelled class ahead by `margin` (CityScapes size: ~4 % of p_t <= 0.7)."""
    B, H, W = cls.shape
    return (margin * F.one_hot(cls.clamp_min(0), C).permute(0, 3, 1, 2).float() + noise * torch.randn(B, C, H, W, generator=g)).contiguous()


def _run(pred, target, **kw):
    """Loss, gradient and the module of both implementations on the same CUDA tensors."""
    import css_b200
    ours = css_b200.ProbOhemCrossEntropy2d(**kw).cuda()
    ref = ohem_ref.ProbOhemCrossEntropy2d(**kw).cuda()
    before = target.clone()
    p1 = pred.detach().clone().requires_grad_(True)
    l1 = ours(p1, target)
    l1.backward()
    assert torch.equal(target, before), "the caller's target was modified"
    p2 = pred.detach().clone().requires_grad_(True)
    l2 = ref(p2, target.clone())
    l2.backward()
    return dict(ours=ours, ref=ref, l1=l1.detach(), l2=l2.detach(), g1=p1.grad, g2=p2.grad)


def _ulp(a, b):
    return (a.view(torch.int32).long() - b.view(torch.int32).long()).abs()


def _check(r, branch, pred=None, target=None, ignore_index=None):
    """branch: 'plain' (no OHEM), 't0' (T = float32(thresh)) or 'select' (T = the min_kept-th smallest p_t)."""
    last, rl = r["ours"].last, r["ref"].last
    T = last["threshold"].item()
    kept = last["p_t"] <= last["threshold"]                  # nan (ignored) compares false
    assert torch.equal(kept, rl["valid_mask"]), f"kept masks differ at {int((kept != rl['valid_mask']).sum())} pixels"
    assert last["num_kept"].item() == int(rl["valid_mask"].sum())
    assert last["num_valid"].item() == int(rl["num_valid"])
    rt = rl["threshold"]
    if branch == "plain":
        assert rt is None and T == math.inf
    else:
        assert rt is not None and isinstance(rt, torch.Tensor) == (branch == "select")
        assert T == torch.as_tensor(rt, dtype=torch.float32).item()
    if pred is not None:                                      # p_t against F.softmax, in ulps
        valid = target != ignore_index
        pt_ref = F.softmax(pred, 1).gather(1, torch.where(valid, target, 0).unsqueeze(1))[:, 0]
        d = int(_ulp(last["p_t"][valid], pt_ref[valid]).max()) if bool(valid.any()) else 0
        print(f"max ulp difference of p_t against F.softmax: {d}")
        assert d == 0
    l1, l2 = r["l1"].item(), r["l2"].item()
    if math.isnan(l2):
        assert math.isnan(l1)
    else:
        np.testing.assert_allclose(l1, l2, rtol=1e-4)
    g1, g2 = r["g1"].cpu().numpy(), r["g2"].cpu().numpy()
    assert np.array_equal(g1 != 0, g2 != 0), "gradient zero patterns differ"
    assert not (g1 != 0).any(axis=1)[~kept.cpu().numpy()].any(), "gradient outside the kept pixels"
    np.testing.assert_allclose(g1, g2, rtol=1e-4, atol=1e-4 * max(float(np.abs(g2).max()), 1e-30) * 1e-3)


# ---- both branches at the CityScapes size ------------------------------------------------------------------------------------

@pytest.mark.parametrize("branch", ["t0", "select"])
def test_cityscapes_full_size(branch):
    from css_b200 import synth
    B, C, H, W = (CITY[k] for k in "BCHW")
    g = synth._gen(31 if branch == "t0" else 32)
    cls = synth.class_map(B, C, H, W, g, ignore_frac=0.05)
    pred = (synth.logits_for(cls, C, g) if branch == "t0" else _confident(cls, C, g)).cuda()
    target = torch.where(cls < 0, torch.full_like(cls, 255), cls).cuda()
    r = _run(pred, target, ignore_index=255, thresh=0.7, min_kept=50000 * B)
    _check(r, branch, pred, target, 255)


# ---- exactness of the selection on crafted logits -----------------------------------------------------------------------------

def _grid(B=2, C=19, H=64, W=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    target = torch.randint(0, C, (B, H, W), generator=g)
    return g, target


def _logits_with_pt_class(target, C, target_logit):
    """Every other logit 0, the labelled one `target_logit` (per pixel tensor or scalar)."""
    B, H, W = target.shape
    oh = F.one_hot(target, C).permute(0, 3, 1, 2).float()
    return (oh * torch.as_tensor(target_logit, dtype=torch.float32).reshape(-1, 1, H, W).expand(B, 1, H, W)).contiguous()


def test_many_ties_at_the_kth_value():
    g, target = _grid()
    B, H, W = target.shape
    tl = torch.full((B, H, W), 8.0)
    tl.view(-1)[: 4000] = 0.0                                 # 4000 pixels with p_t = 1/19 exactly alike
    tl.view(-1)[4000: 4050] = -3.0                            # 50 below them
    pred = _logits_with_pt_class(target, 19, tl).cuda()
    r = _run(pred, target.cuda(), ignore_index=255, thresh=0.01, min_kept=100)
    _check(r, "select")
    assert r["ours"].last["num_kept"].item() == 4050


@pytest.mark.parametrize("where", ["equal", "above", "below"])
def test_kth_at_and_next_to_thresh(where):
    g, target = _grid(seed=1)
    B, H, W = target.shape
    tl = torch.full((B, H, W), 8.0)
    tl.view(-1)[:100] = -3.0
    tl.view(-1)[100:400] = 2.5
    pred = _logits_with_pt_class(target, 19, tl).cuda()
    v = F.softmax(pred, 1).gather(1, target.cuda().unsqueeze(1)).view(-1)[100].item()     # the kth value, a float32
    thresh = {"equal": v, "above": float(np.nextafter(np.float32(v), np.float32(1))),
              "below": float(np.nextafter(np.float32(v), np.float32(0)))}[where]
    r = _run(pred, target.cuda(), ignore_index=255, thresh=thresh, min_kept=250)
    _check(r, "select" if where == "below" else "t0")
    assert r["ours"].last["num_kept"].item() == 400
    assert r["ours"].last["threshold"].item() == (v if where != "above" else np.float32(thresh))


def test_kth_saturated_at_one():
    g, target = _grid(seed=2)
    B, H, W = target.shape
    tl = torch.full((B, H, W), 100.0)                         # p_t == 1.0 exactly
    tl.view(-1)[:20] = 0.5
    pred = _logits_with_pt_class(target, 19, tl).cuda()
    r = _run(pred, target.cuda(), ignore_index=255, thresh=0.7, min_kept=1000)
    _check(r, "select")
    assert r["ours"].last["threshold"].item() == 1.0 and r["ours"].last["num_kept"].item() == B * H * W


@pytest.mark.parametrize("thresh", [0.7, -1.0])
def test_pt_underflow_to_zero(thresh):
    g, target = _grid(seed=3)
    B, H, W = target.shape
    tl = torch.full((B, H, W), 3.0)
    tl.view(-1)[:500] = -200.0                                # p_t == 0.0
    pred = _logits_with_pt_class(target, 19, tl).cuda()
    r = _run(pred, target.cuda(), ignore_index=255, thresh=thresh, min_kept=100)
    _check(r, "t0" if thresh > 0 else "select")
    if thresh < 0:
        assert r["ours"].last["threshold"].item() == 0.0 and r["ours"].last["num_kept"].item() == 500


@pytest.mark.parametrize("which", ["num_valid", "num_valid+1", "one", "zero"])
def test_min_kept_edges(which):
    from css_b200 import synth
    g = synth._gen(4)
    cls = synth.class_map(2, 19, 48, 40, g, ignore_frac=0.2, block=4)
    pred = synth.logits_for(cls, 19, g).cuda()
    target = torch.where(cls < 0, torch.full_like(cls, 255), cls).cuda()
    nv = int((cls >= 0).sum())
    mk = {"num_valid": nv, "num_valid+1": nv + 1, "one": 1, "zero": 0}[which]
    r = _run(pred, target, ignore_index=255, thresh=0.7, min_kept=mk)
    _check(r, {"num_valid": "select", "num_valid+1": "plain", "one": "t0", "zero": "plain"}[which])


def test_all_pixels_ignored():
    g, target = _grid(seed=5)
    pred = torch.randn(2, 19, 64, 64, generator=g).cuda()
    r = _run(pred, torch.full_like(target, 255).cuda(), ignore_index=255, thresh=0.7, min_kept=100)
    _check(r, "plain")
    assert math.isnan(r["l1"].item()) and not r["g1"].any()
    assert r["ours"].last["num_valid"].item() == 0 and r["ours"].last["num_kept"].item() == 0


@pytest.mark.parametrize("ignore_index", [-1, 255])
@pytest.mark.parametrize("confident", [False, True])
def test_ignore_index_values(ignore_index, confident):
    from css_b200 import synth
    g = synth._gen(6)
    cls = synth.class_map(3, 19, 65, 67, g, ignore_frac=0.1, block=4)
    pred = (_confident(cls, 19, g) if confident else synth.logits_for(cls, 19, g)).cuda()
    target = torch.where(cls < 0, torch.full_like(cls, ignore_index), cls).cuda()
    r = _run(pred, target, ignore_index=ignore_index, thresh=0.7, min_kept=3000)
    _check(r, "select" if confident else "t0")


@pytest.mark.parametrize("confident", [False, True])
def test_class_weights(confident):
    from css_b200 import synth
    g = synth._gen(7)
    cls = synth.class_map(2, 19, 129, 97, g, ignore_frac=0.1, block=4)
    pred = (_confident(cls, 19, g) if confident else synth.logits_for(cls, 19, g)).cuda()
    target = torch.where(cls < 0, torch.full_like(cls, 255), cls).cuda()
    r = _run(pred, target, ignore_index=255, thresh=0.7, min_kept=2000, use_weight=True)
    _check(r, "select" if confident else "t0")


@pytest.mark.parametrize("C", [7, 21])
@pytest.mark.parametrize("confident", [False, True])
def test_other_class_counts(C, confident):
    from css_b200 import synth
    g = synth._gen(8 + C)
    cls = synth.class_map(2, C, 96, 111, g, ignore_frac=0.1, block=4)
    pred = (_confident(cls, C, g) if confident else synth.logits_for(cls, C, g)).cuda()
    target = torch.where(cls < 0, torch.full_like(cls, 255), cls).cuda()
    r = _run(pred, target, ignore_index=255, thresh=0.7, min_kept=1500)
    _check(r, "select" if confident else "t0", pred, target, 255)


# ---- CUDA graphs and other properties ---------------------------------------------------------------------------------------

def _city_batch(seed, confident, B=2, H=257, W=259, C=19):
    from css_b200 import synth
    g = synth._gen(seed)
    cls = synth.class_map(B, C, H, W, g, ignore_frac=0.05)
    pred = _confident(cls, C, g) if confident else synth.logits_for(cls, C, g)
    return pred.cuda(), torch.where(cls < 0, torch.full_like(cls, 255), cls).cuda()


def test_graph_capture_replays_on_new_inputs():
    import css_b200
    kw = dict(ignore_index=255, thresh=0.7, min_kept=20000)
    crit = css_b200.ProbOhemCrossEntropy2d(**kw).cuda()
    pa, ta = _city_batch(40, False)
    pb, tb = _city_batch(41, True)
    eager = []
    for p, t in ((pa, ta), (pb, tb)):
        leaf = p.clone().requires_grad_(True)
        loss = crit(leaf, t)
        (gr,) = torch.autograd.grad(loss, leaf)
        eager.append((loss.clone(), gr.clone(), crit.last["threshold"].clone(), crit.last["num_kept"].clone()))
    static_pred = pa.clone().requires_grad_(True)
    static_t = ta.clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            torch.autograd.grad(crit(static_pred, static_t), static_pred)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss = crit(static_pred, static_t)
        (grad,) = torch.autograd.grad(loss, static_pred)
    last = crit.last
    for (p, t), (el, eg, eT, ek) in zip(((pb, tb), (pa, ta), (pb, tb)), (eager[1], eager[0], eager[1])):
        with torch.no_grad():
            static_pred.copy_(p)
            static_t.copy_(t)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(loss, el) and torch.equal(grad, eg)
        assert torch.equal(last["threshold"], eT) and torch.equal(last["num_kept"], ek)
    assert eager[0][2].item() == np.float32(0.7) and eager[1][2].item() > np.float32(0.7)       # both branches replayed


def test_two_calls_bit_identical_and_channels_last():
    import css_b200
    pred, target = _city_batch(42, True)
    crit = css_b200.ProbOhemCrossEntropy2d(ignore_index=255, thresh=0.7, min_kept=20000, use_weight=True).cuda()
    outs = []
    for p in (pred, pred, pred.contiguous(memory_format=torch.channels_last)):
        leaf = p.clone(memory_format=torch.preserve_format).requires_grad_(True)
        loss = crit(leaf, target)
        loss.backward()
        outs.append((loss.detach(), leaf.grad.contiguous(), crit.last["threshold"].clone(), crit.last["num_kept"].clone()))
    assert pred.contiguous(memory_format=torch.channels_last).is_contiguous(memory_format=torch.channels_last)
    for o in outs[1:]:
        assert all(torch.equal(a, b) for a, b in zip(outs[0], o))


def test_out_of_range_labels_are_ignored():
    pred, target = _city_batch(43, True, B=2, H=97, W=99)
    bad = target.clone()
    bad.view(-1)[::7] = 19
    bad.view(-1)[3::11] = -5
    bad.view(-1)[5::13] = 1000
    import css_b200
    crit = css_b200.ProbOhemCrossEntropy2d(ignore_index=255, thresh=0.7, min_kept=2000).cuda()
    leaf = pred.clone().requires_grad_(True)
    loss = crit(leaf, bad)
    loss.backward()
    torch.cuda.synchronize()
    clean = torch.where((bad < 0) | (bad >= 19), torch.full_like(bad, 255), bad)
    r = _run(pred, clean, ignore_index=255, thresh=0.7, min_kept=2000)
    assert torch.equal(loss, r["l1"]) and torch.equal(leaf.grad, r["g1"])
    _check(r, "select")
