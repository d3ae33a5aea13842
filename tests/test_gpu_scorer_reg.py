"""The default fp32 gradient scorer (path 0, score_ce_kernel on whole-warp rows) beyond the kernel matrix's cases: the models'
temperatures, more than one 32-id batch per warp, draws fed back bit-identical to the same draws made on the fly, the bench
shapes, and agreement with the register / bulk-copy hybrid on 8-lane groups (path 2) on the same draws.

Every case is checked against the float64 reference (oracle/f64_ref.py) with the kernel matrix's helpers and tolerances, and
the profiler confirms which instantiation ran.
"""
import numpy as np
import pytest
import torch

from tests import test_gpu_kernel_matrix as M

pytestmark = pytest.mark.gpu
lib = M.lib                               # the matrix module's fixture: FFMA2 rep pass, scorer path reset afterwards

TEMPS = (0.5, 0.25, 0.1, 0.0241, 0.0240)  # the models' temperatures and both sides of the fixed-reference switch


def reg_kernel(fix, fed):
    return M.scorer_kernel("grad-f32-reg", fix, fed)


def run_reg(lib, rep, label, mask, prob, protos, kw, seed, indices=None):
    """One Contrast_Loss forward + backward on path 0."""
    return M.run_loss(lib, "grad-f32-reg", rep, label, mask, prob, protos, kw, seed, indices=indices)


def check_vs_path2(lib, rep, label, mask, prob, protos, kw, seed, indices, loss, grad, crit):
    """Same draws on the 8-lane-group hybrid: same anchor pixels, loss to rel 2e-6, gradient as in test_scorer_paths_agree."""
    l0, g0, c0, _, _ = M.run_loss(lib, "grad-f32-bulk", rep, label, mask, prob, protos, kw, seed, indices=indices)
    assert torch.equal(crit.last["anchor_px"], c0.last["anchor_px"])
    assert abs(loss.item() - l0.item()) <= 2e-6 * abs(l0.item())
    g0 = g0.cpu().numpy()
    assert np.abs(g0).max() > 0
    np.testing.assert_allclose(grad.cpu().numpy(), g0, rtol=1e-5, atol=2e-6 * np.abs(g0).max())


@pytest.mark.parametrize("temp", TEMPS)
def test_reg_scorer(lib, temp):
    """Drawn on the fly, then the same draws fed: both instantiations against float64, fed == fly bit for bit, and path 0."""
    B2, C, h, w, Q, Nn, seed = 2, 7, 19, 23, 12, 100, 31
    rep, label, mask, prob, protos = M.scorer_inputs(B2, C, h, w, seed)
    kw = dict(num_queries=Q, num_negatives=Nn, temp=temp, strong_threshold=0.97, alpha=0.99)
    fix = temp > M.FIX_SWITCH
    (loss, grad, crit, p0, p), names = M.launched(lambda: run_reg(lib, rep, label, mask, prob, protos, kw, seed))
    M.assert_launched([reg_kernel(fix, False)], names)
    a, n = crit.sample_indices(seed, 0)
    M.check_against_f64("grad-f32-reg", loss, grad, crit, p0, p, rep, label, mask, kw, a, n, "scorer reg")
    (loss_f, grad_f, crit_f, p0_f, p_f), names = M.launched(lambda: run_reg(lib, rep, label, mask, prob, protos, kw, seed, (a, n)))
    M.assert_launched([reg_kernel(fix, True)], names)
    M.check_against_f64("grad-f32-reg", loss_f, grad_f, crit_f, p0_f, p_f, rep, label, mask, kw, a, n, "scorer reg")
    assert loss_f.item() == loss.item()
    assert torch.equal(grad_f, grad)
    check_vs_path2(lib, rep, label, mask, prob, protos, kw, seed, (a, n), loss, grad, crit)


@pytest.mark.parametrize("Nn", [129, 160, 512])
def test_reg_scorer_candidate_counts(lib, Nn):
    """More than 32 negatives per warp: a second id batch with a single candidate (129), a full second batch (160), and the
    bench's 512 (four full batches per warp)."""
    B2, C, h, w, Q, seed = 2, 5, 13, 15, 9, 5 + Nn
    rep, label, mask, prob, protos = M.scorer_inputs(B2, C, h, w, seed)
    kw = dict(num_queries=Q, num_negatives=Nn, temp=0.5, strong_threshold=0.97, alpha=0.99)
    (loss, grad, crit, p0, p), names = M.launched(lambda: run_reg(lib, rep, label, mask, prob, protos, kw, seed))
    M.assert_launched([reg_kernel(True, False)], names)
    a, n = crit.sample_indices(seed, 0)
    M.check_against_f64("grad-f32-reg", loss, grad, crit, p0, p, rep, label, mask, kw, a, n, "scorer reg")
    check_vs_path2(lib, rep, label, mask, prob, protos, kw, seed, (a, n), loss, grad, crit)


@pytest.mark.parametrize("B2,C,h,w", [(16, 21, 81, 81), (8, 19, 193, 193)], ids=["voc81", "city193"])
def test_reg_scorer_bench_shapes(lib, B2, C, h, w):
    """The shapes bench.py times: Q=256, Nn=512 on VOC 81x81 (B2=16) and CityScapes 193x193 (B2=8)."""
    Q, Nn, seed = 256, 512, 2024 + C
    rep, label, mask, prob, protos = M.scorer_inputs(B2, C, h, w, seed)
    kw = dict(num_queries=Q, num_negatives=Nn, temp=0.5, strong_threshold=0.97, alpha=0.99)
    (loss, grad, crit, p0, p), names = M.launched(lambda: run_reg(lib, rep, label, mask, prob, protos, kw, seed))
    M.assert_launched([reg_kernel(True, False)], names)
    a, n = crit.sample_indices(seed, 0)
    M.check_against_f64("grad-f32-reg", loss, grad, crit, p0, p, rep, label, mask, kw, a, n, "scorer reg bench")
    check_vs_path2(lib, rep, label, mask, prob, protos, kw, seed, (a, n), loss, grad, crit)
