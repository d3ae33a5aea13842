"""Every compiled kernel specialisation the suite drives, each compared with a float64 reference (oracle/f64_ref.py).

Each case names the instantiations it must launch ("rep_pass_kernel<7, false, float, false>").  The case runs under
torch.profiler with CUDA activities (in memory, no trace file) and fails unless every declared kernel is among the launched
ones, so a dispatch change that sends a case to another specialisation cannot pass silently.  tests/test_kernel_manifest.py
checks that these declarations, together with its short list of kernels driven by other tests, cover every kernel compiled
into libcss_b200.so.  The declarations below build without a GPU; the tests need one.

Tolerances are those of DESIGN.md section 2, measured against float64: similarities / probabilities abs 1e-6, norms rel 1e-6,
confidences abs 2e-6, losses and gradients rel 1e-4 (gradient elements with 2e-5 of the largest element as absolute slack,
as in test_gpu_fullsize.py).  At the models' temperatures (0.25, 0.1) a probability or confidence bound is the larger of
these and the error of torch's own float32 statements on the same inputs (f32_bound).  Set CSS_B200_F64_REPORT=<file> to
write the largest error of each kernel family as JSON.
"""
import json
import math
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.helpers import TAU

pytestmark = pytest.mark.gpu

F32, BF16 = "float", "__nv_bfloat16"
RTOL = 1e-4
TEMP = 0.5


def _b(v):
    return "true" if v else "false"


def rep_kernel(ng, rows, t, t1=False):
    return f"rep_pass_kernel<{ng}, {_b(rows)}, {t}, {_b(t1)}>"


def normalise(name):
    """Kernel name without the return type and the parameter list: 'void f<1, true>(float*, int)' -> 'f<1, true>'."""
    name = re.sub(r"^void\s+", "", name.strip())
    return name.split("(", 1)[0].strip()


# ---------------------------------------------------------------------------------------------------------------------------
# declarations (no CUDA needed)
# ---------------------------------------------------------------------------------------------------------------------------
REP_CLASSES = (1, 4, 7, 12, 13, 16, 19, 21, 22, 24, 25, 28, 32)     # NG = ceil(C / 4) = 1..8, with and without a ragged group
REP_SHAPES = ("ragged", "persistent")


def _rep_cases():
    out = []
    for C in REP_CLASSES:
        ng, t1 = (C + 3) // 4, C == 21
        for mode in ("cos", "softmax_rows"):
            for t in (F32, BF16):
                for shape in REP_SHAPES:
                    ks = ["proto_prep_kernel", rep_kernel(ng, mode != "cos", t, t1)]
                    if t == BF16:                                # compared bit for bit with the fp32 kernel on rep.float()
                        ks.append(rep_kernel(ng, mode != "cos", F32, t1))
                    out.append(pytest.param(C, mode, t, shape, ks, id=f"C{C}-{mode}-{'f32' if t == F32 else 'bf16'}-{shape}"))
    for t in (F32, BF16):
        for shape in REP_SHAPES:
            ks = [rep_kernel(0, True, t)] + ([rep_kernel(0, True, F32)] if t == BF16 else [])
            out.append(pytest.param(0, "rows_only", t, shape, ks, id=f"rows_only-{'f32' if t == F32 else 'bf16'}-{shape}"))
    return out


REP_CASES = _rep_cases()

# (C, h, w, H, W, temp, tile, kernel); tile: "staged" (<= 48 KB of shared memory), "optin" (> 48 KB, the opt-in attribute),
# "global" (the footprint exceeds 96 KB: taps read from global memory).  Every scale (in-1)/(out-1) is a power of two, so
# fp32 source coordinates are exact and the float64 F.interpolate weighs the same taps: ATen computes the coordinates of a
# float32 tensor in fp32, which at other ratios moves a tap by up to ~1e-5 and would be measured here as kernel error.
UPSAMPLE_CASES = [
    pytest.param(21, 41, 41, 161, 161, 0.5, "staged", "upsample_label_fuse_kernel<true, 21>", id="C21-staged"),
    pytest.param(19, 49, 33, 193, 129, 0.3, "staged", "upsample_label_fuse_kernel<true, 19>", id="C19-staged"),
    pytest.param(21, 41, 41, 161, 161, 0.25, "staged", "upsample_label_fuse_kernel<true, 21>", id="C21-staged-t0.25"),
    pytest.param(21, 41, 41, 161, 161, 0.1, "staged", "upsample_label_fuse_kernel<true, 21>", id="C21-staged-t0.1"),
    pytest.param(19, 49, 33, 193, 129, 0.25, "staged", "upsample_label_fuse_kernel<true, 19>", id="C19-staged-t0.25"),
    pytest.param(19, 49, 33, 193, 129, 0.1, "staged", "upsample_label_fuse_kernel<true, 19>", id="C19-staged-t0.1"),
    pytest.param(7, 33, 31, 129, 121, 0.5, "staged", "upsample_label_fuse_kernel<true, 0>", id="C7-staged"),
    pytest.param(32, 20, 21, 77, 81, 0.7, "staged", "upsample_label_fuse_kernel<true, 0>", id="C32-staged"),
    pytest.param(21, 40, 50, 40, 50, 0.5, "optin", "upsample_label_fuse_kernel<true, 21>", id="C21-optin"),
    pytest.param(19, 40, 50, 40, 50, 0.3, "optin", "upsample_label_fuse_kernel<true, 19>", id="C19-optin"),
    pytest.param(5, 40, 50, 40, 50, 0.5, "optin", "upsample_label_fuse_kernel<true, 0>", id="C5-optin"),
    pytest.param(21, 129, 97, 33, 25, 0.5, "global", "upsample_label_fuse_kernel<false, 0>", id="C21-global"),
    pytest.param(1, 97, 129, 25, 33, 0.5, "global", "upsample_label_fuse_kernel<false, 0>", id="C1-global"),
]


def scorer_kernel(variant, fix, fed):
    """The kernel css_score_ce picks for a variant (css_score.cu:861-891)."""
    return {"grad-f32-reg": f"score_ce_kernel<true, false, true, {_b(fix)}, float>",
            "grad-f32-ring": f"score_ce_ring_kernel<{_b(fix)}, {_b(fed)}, 2, 4>",
            "grad-f32-bulk": f"score_ce_bulk_kernel<{_b(fix)}, {_b(fed)}, 2, 1, 4>",
            "grad-bf16": f"score_ce_kernel<true, false, true, {_b(fix)}, {BF16}>",
            "nograd-f32": f"score_ce_kernel<false, true, false, {_b(fix)}, float>",
            "nograd-bf16": f"score_ce_kernel<false, false, false, {_b(fix)}, {BF16}>"}[variant]


SCORER_VARIANTS = ("grad-f32-reg", "grad-f32-ring", "grad-f32-bulk", "grad-bf16", "nograd-f32", "nograd-bf16")
SCORER_PATH = {"grad-f32-reg": 0, "grad-f32-ring": 1, "grad-f32-bulk": 2}
FIX_SWITCH = 2 * 1.4426950408889634 / 120.0          # css_score.cu:863: fixed-reference softmax above this temperature


# the rest of a Contrast_Loss forward: selection, class sums, prototype EMA + class CDF, Philox offset, loss reduction (the
# updated prototypes and the loss are compared with float64 too)
LOSS_CHAIN = ("select_classify_kernel", "select_scan_kernel", "select_scatter_kernel", "class_reduce_kernel", "proto_ema_kernel",
              "class_cdf_kernel", "draw_offset_kernel", "loss_reduce_kernel")


def _scorer_cases():
    out = []
    for v in SCORER_VARIANTS:
        for temp in (0.5, 0.02):
            for draws in ("fly", "fed"):
                ks = [scorer_kernel(v, temp > FIX_SWITCH, draws == "fed")] + list(LOSS_CHAIN)
                ks.append(f"class_sums_kernel<{BF16 if v.endswith('bf16') else F32}>")
                if v.startswith("grad"):
                    ks.append("grad_slab_kernel")
                if v.startswith("nograd"):                  # compared with the path-0 gradient kernel's loss on the same draws
                    ks.append(scorer_kernel("grad-f32-reg", temp > FIX_SWITCH, False))
                out.append(pytest.param(v, temp, draws, ks, id=f"{v}-t{temp}-{draws}"))
    return out


SCORER_CASES = _scorer_cases()
NN_EDGE_CASES = [pytest.param(v, nn, [scorer_kernel(v, True, False)], id=f"{v}-Nn{nn}")
                 for v in ("grad-f32-reg", "grad-f32-ring", "grad-f32-bulk", "nograd-f32") for nn in (1, 31, 32, 33)]
TEMP_SWITCH_CASES = [pytest.param(t, [scorer_kernel("grad-f32-reg", t > FIX_SWITCH, False),
                                      scorer_kernel("nograd-f32", t > FIX_SWITCH, False)], id=f"t{t}")
                     for t in (0.0240, 0.0241)]
BENCH_CASES = [pytest.param(16, 21, 81, 81, [scorer_kernel("grad-f32-bulk", True, False)], id="voc81"),
               pytest.param(8, 19, 193, 193, [scorer_kernel("grad-f32-bulk", True, False)], id="city193")]
ROWS_VERIFY_KERNELS = [f"rows_verify_kernel<{BF16}>", rep_kernel(0, True, BF16)]
ATL_CASES = [pytest.param(C, B, ["atl_forward_kernel<0>", "atl_finalize_kernel", "atl_backward_kernel<0>"], id=f"C{C}-B{B}")
             for C in (2, 7, 32) for B in (1, 9, 17, 256)]
PEER_WORLDS = (3, 5, 9)


def peer_kernel(world):
    return f"stats_allreduce_kernel<{2 if world <= 2 else 4 if world <= 4 else 8 if world <= 8 else 16}>"


PEER_KERNELS = [peer_kernel(w) for w in PEER_WORLDS]

# the models' own temperatures: Model_mix 0.25, Model_cross 0.1 (models.py:93,116); an error in a cosine reaches their
# probabilities scaled by 1/temp
MODEL_TEMPS = (0.25, 0.1)
REP_TEMP_CASES = [pytest.param(C, t, ["proto_prep_kernel", rep_kernel((C + 3) // 4, True, F32, C == 21)], id=f"C{C}-t{t}")
                  for C in REP_CLASSES for t in MODEL_TEMPS]
SIM_MODES = ((None, "cos"), (0.5, "t0.5"), (0.25, "t0.25"), (0.1, "t0.1"))     # (softmax temperature or None = cosine, id)

# channels-last rep pass (css_sim_tc.cu rep_pass_nhwc_kernel<NP>: NP = 3 for C <= 24, 4 above, with padded class columns)
NHWC_CLASSES = (1, 5, 19, 21, 24, 25, 31, 32)
NHWC_SHAPES = ("one_tile", "exact128", "ragged", "sub_wave", "city193")


def nhwc_kernel(C):
    return f"rep_pass_nhwc_kernel<{3 if C <= 24 else 4}>"


NHWC_CASES = [pytest.param(C, shape, t, ["proto_prep_tc_kernel", nhwc_kernel(C)], id=f"C{C}-{shape}-{tid}")
              for C in NHWC_CLASSES for shape in NHWC_SHAPES for t, tid in SIM_MODES]
NHWC_ALIGN_CASES = [pytest.param(4, ["proto_prep_tc_kernel", nhwc_kernel(21)], id="offset16B-channels_last"),
                    pytest.param(1, ["proto_prep_kernel", rep_kernel(6, True, F32, True)], id="offset4B-nchw_copy")]
NHWC_REFRESH_KERNELS = ["rows_verify_rm_kernel", nhwc_kernel(1)]
NHWC_LOSS_KERNELS = ["rows_verify_rm_kernel", nhwc_kernel(1), "grad_rows_kernel"]

# NCHW tensor-core rep pass (css_sim_tc.cu rep_pass_tc_kernel<ROWS, NP>, opt-in with css_set_rep_pass_path(1)); the map at a
# storage offset of 0..3 floats: 1..3 put every plane window's start off 16 bytes (the base16 lead-in) and send the first
# plane through the loader's per-lane copy
TC_CLASSES = (1, 5, 21, 24, 25, 32)
TC_SHAPES = {"hw63": (1, 7, 9), "hw128": (2, 8, 16), "hw129": (3, 3, 43), "hw510": (2, 17, 30), "city193": (8, 193, 193)}
TC_OFFSETS = (0, 1, 2, 3)


def tc_kernels(C, rows):
    return ["proto_prep_tc_kernel", f"rep_pass_tc_kernel<{_b(rows)}, {3 if C <= 24 else 4}>"]


TC_CASES = ([pytest.param(C, "hw510", off, t, tc_kernels(C, t is not None), id=f"C{C}-hw510-off{off}-{tid}")
             for C in TC_CLASSES for off in TC_OFFSETS for t, tid in SIM_MODES]
            + [pytest.param(C, shape, off, t, tc_kernels(C, t is not None), id=f"C{C}-{shape}-off{off}-{tid}")
               for shape in ("hw63", "hw128", "hw129", "city193") for off in TC_OFFSETS for C, t, tid in ((21, 0.1, "t0.1"), (25, None, "cos"))])


def declared_kernels():
    """Every instantiation some case of this module asserts it launches."""
    out = set()
    for cases in (REP_CASES, REP_TEMP_CASES, SCORER_CASES, NN_EDGE_CASES, TEMP_SWITCH_CASES, BENCH_CASES, ATL_CASES, NHWC_CASES,
                  NHWC_ALIGN_CASES, TC_CASES):
        for p in cases:
            out.update(p.values[-1])
    out.update(p.values[-1] for p in UPSAMPLE_CASES)
    out.update(ROWS_VERIFY_KERNELS)
    out.update(PEER_KERNELS)
    out.update(NHWC_REFRESH_KERNELS)
    out.update(NHWC_LOSS_KERNELS)
    out.add(scorer_kernel("grad-f32-reg", False, False))           # test_scorer_anti_aligned_candidates (online-max side)
    out.add(scorer_kernel("grad-f32-reg", True, False))
    return out


# ---------------------------------------------------------------------------------------------------------------------------
# running and measuring
# ---------------------------------------------------------------------------------------------------------------------------
MAX_ERR = {}


def record(family, err):
    MAX_ERR[family] = max(MAX_ERR.get(family, 0.0), float(err))


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    path = os.environ.get("CSS_B200_F64_REPORT")
    if path and MAX_ERR:
        with open(path, "w") as f:
            json.dump(dict(sorted(MAX_ERR.items())), f, indent=1)


def launched(fn):
    """Runs fn() under the CUDA profiler; returns (fn's result, set of normalised kernel names launched)."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = {normalise(e.name) for e in prof.events() if e.device_type == DeviceType.CUDA}
    kernels = {n for n in names if not n.startswith(("Memcpy", "Memset"))}
    assert kernels, "the profiler recorded no kernel launches at all: cannot check which specialisations ran"
    return out, kernels


def assert_launched(declared, names):
    missing = sorted(set(declared) - names)
    assert not missing, f"declared kernels not launched: {missing}; launched: {sorted(names)}"


@pytest.fixture
def lib():
    from css_b200 import _lib
    lib = _lib.load()
    lib.css_set_rep_pass_path(0)              # the FFMA2 kernels of css_sim.cu (the tensor-core side has its own tests)
    yield lib
    lib.css_set_rep_pass_path(-1)
    lib.css_set_scorer_path(-1)


def rel_norm_err(got, ref):
    return float(torch.linalg.vector_norm((got.double() - ref).ravel()) / torch.linalg.vector_norm(ref.ravel()).clamp_min(1e-300))


def check_grad(got, ref, rtol=RTOL, family=None):
    """Support identical, elementwise rel rtol with 2e-5 of the largest element as absolute slack, norm-wise rel < rtol."""
    got = got.double()
    slack = 2e-5 * float(ref.abs().max())
    assert not ((got != 0) & (ref == 0)).any(), "gradient on pixels that are no anchor"
    # a query whose softmax is one-hot to fp32 precision (temp 0.02: logit gaps of ~100) has a gradient below the resolution of
    # the fp32 terms it is the difference of, and the kernel returns exact zeros there (as the fp32 oracle does); float64 keeps
    # values of ~e^-100.  Such zeros are accepted only below the absolute slack.
    lost = (got == 0) & (ref != 0)
    assert not (lost & (ref.abs() > slack)).any(), "gradient support differs from float64"
    excess = ((got - ref).abs() - rtol * ref.abs()).max().item()
    assert excess <= slack, f"gradient: max |err| - rtol |ref| = {excess:.3e} > {slack:.3e}"
    err = rel_norm_err(got, ref)
    assert err < rtol, f"gradient norm-wise relative error {err:.2e}"
    if family:
        record(family + " grad (norm-wise rel)", err)
        record(family + " grad: largest |float64| where the kernel gives 0", ref.abs()[lost].max() if lost.any() else 0.0)


def check_loss(got, ref, rtol=RTOL, family=None):
    err = abs(float(got.detach()) - float(ref)) / abs(float(ref))
    assert err <= rtol, f"loss {float(got)!r} vs float64 {float(ref)!r}: rel {err:.2e}"
    if family:
        record(family + " loss (rel)", err)


def f32_bound(bound, torch_f32_err, family):
    """At the models' temperatures the bound on a probability or confidence is the larger of the fixed one and the error of
    torch's own float32 statements on the same inputs, measured against the same float64 reference (DESIGN.md section 2)."""
    record(family, torch_f32_err)
    return max(bound, torch_f32_err)


def torch_f32_prob(x, protos, temp):
    """ddp_model.py:147-154 as the reference runs it in float32: F.normalize, mm (no TF32), softmax."""
    B, D, h, w = x.shape
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        sim = F.normalize(x.float().permute(0, 2, 3, 1).reshape(-1, D), dim=-1) @ F.normalize(protos.float(), dim=-1).T
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return torch.softmax(sim / temp, dim=1).reshape(B, h, w, -1).permute(0, 3, 1, 2)


def check_sim_map(out, x, protos, temp, family):
    """A cosine map (temp None) or softmax(cos / temp) against float64: abs 1e-6 (at the models' temperatures, see f32_bound).
    x carries rich_map's content: a zero prototype row and a zero-norm pixel give exact zeros in a cosine map."""
    from oracle import f64_ref as R
    C = protos.shape[0]
    if temp is None:
        err = (out.double() - R.cos_sim_map(x, protos)).abs().max().item()
        record(family + " sim", err)
        assert err <= 1e-6, f"cos: max abs error {err:.3e} vs float64"
        if C > 1:
            assert (out[:, C // 2] == 0).all(), "the zero prototype row has a non-zero similarity"
        assert (out[0, :, 0, 1] == 0).all(), "the zero-norm pixel has a non-zero similarity"
        return
    ref = R.proto_softmax_sim(x, protos, temp)
    err = (out.double() - ref).abs().max().item()
    bound = 1e-6
    if temp in MODEL_TEMPS:
        bound = f32_bound(bound, (torch_f32_prob(x, protos, temp).double() - ref).abs().max().item(), f"torch float32 prob t{temp}")
    record(f"{family} prob t{temp}" if temp in MODEL_TEMPS else family + " prob", err)
    assert err <= bound, f"softmax t{temp}: max abs error {err:.3e} vs float64 (bound {bound:.3e})"


def check_norms(norms, x, family):
    nref = torch.linalg.vector_norm(x.double(), dim=1).reshape(-1)
    assert norms[1].item() == 0.0                                      # rich_map's zero-norm pixel (0, 0, 1)
    rel = ((norms.double() - nref).abs() / nref.clamp_min(1e-300)).max().item()
    record(family + " norms (rel)", rel)
    assert rel <= 1e-6, f"norms: max rel error {rel:.3e} vs float64"


def rich_map(B, h, w, C, seed):
    """A [B,256,h,w] map and [C,256] prototypes on the GPU with the content where a similarity kernel can go wrong: a zero-norm
    pixel, a zero prototype row (C > 1), a pixel that is a multiple of the last prototype (cos = 1), a pixel with one channel
    ~1e3 and the rest ~1e-3.  Normal values nearly always have some of their low 13 mantissa bits set, the bits a TF32 operand
    drops, so the lo term of the tensor-core kernels' hi/lo split carries weight."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(B, 256, h, w, generator=g, device="cuda")
    assert ((x.view(torch.int32) & 0x1FFF) != 0).float().mean().item() > 0.99
    protos = 0.5 * torch.randn(C, 256, generator=g, device="cuda")
    if C > 1:
        protos[C // 2] = 0
    px = x.view(B, 256, h * w)
    px[0, :, 1] = 0
    px[0, :, 2] = 3 * protos[C - 1]
    px[0, :, 3] *= 1e-3
    px[0, 7, 3] = 1000.123
    return x, protos


# ---------------------------------------------------------------------------------------------------------------------------
# rep pass (css_sim.cu rep_pass_kernel: NG 1..8 x ROWS x fp32 / bf16, the rows-only pass)
# ---------------------------------------------------------------------------------------------------------------------------
def rep_shape(shape):
    if shape == "ragged":
        return 3, 17, 29                      # h*w = 493 odd, N = 1479 not a multiple of 128
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    cap = 4 * sms * 128                       # css_sim.cu:262-265: grid capped at 4 CTAs/SM of 128 pixels
    h = 199
    w = math.ceil(1.5 * cap / (2 * h)) | 1    # N ~ 1.5 x cap: every CTA runs a second grid-stride round
    assert 2 * h * w > cap
    return 2, h, w


@pytest.mark.parametrize("C,mode,dtype,shape,kernels", REP_CASES)
def test_rep_pass(lib, C, mode, dtype, shape, kernels):
    import css_b200
    from oracle import f64_ref as R
    B, h, w = rep_shape(shape)
    g = torch.Generator().manual_seed(1000 * C + h)
    rep = torch.randn(B, 256, h, w, generator=g)
    rep[0, :, 0, 1] = 0                                                # a zero-norm pixel
    rep = rep.cuda().to(torch.bfloat16 if dtype == BF16 else torch.float32)
    protos = None
    if C:
        protos = 0.5 * torch.randn(C, 256, generator=g)
        if C > 1:
            protos[C // 2] = 0                                         # a zero prototype row
        protos = protos.cuda()

    def run(x):
        if mode == "cos":
            return css_b200.ops.cos_sim_map(x, protos), None, None
        if mode == "softmax_rows":
            p = css_b200.ops.proto_softmax_sim(x, protos, TEMP)
            return p, p._css_rows.rows, p._css_rows.norms
        rows, norms = css_b200.ops.rep_rows(x)
        return None, rows, norms

    (first, second), names = launched(lambda: _run_pair(run, rep, dtype))
    assert_launched(kernels, names)
    (out, rows, norms), (out32, rows32, norms32) = first, second
    x32 = rep.float()
    if dtype == BF16:                                             # exact widening: bit-identical to the fp32 kernel
        if out is not None:
            assert torch.equal(out, out32)
        if rows is not None:
            assert rows.dtype == torch.bfloat16 and torch.equal(rows.float(), rows32) and torch.equal(norms, norms32)
    if out32 is not None:
        ref = R.cos_sim_map(x32, protos) if mode == "cos" else R.proto_softmax_sim(x32, protos, TEMP)
        err = (out32.double() - ref).abs().max().item()
        record("rep_pass sim" if mode == "cos" else "rep_pass prob", err)
        assert err <= 1e-6, f"{mode}: max abs error {err:.3e} vs float64"
        if C > 1 and mode == "cos":
            assert (out32[:, C // 2] == 0).all()
    if rows32 is not None:
        assert torch.equal(rows32, x32.permute(0, 2, 3, 1).reshape(-1, 256))
        nref = torch.linalg.vector_norm(x32.double(), dim=1).reshape(-1)
        assert norms32[1].item() == 0.0                              # pixel (0, 0, 1)
        rel = ((norms32.double() - nref).abs() / nref.clamp_min(1e-300)).max().item()
        record("rep_pass norms (rel)", rel)
        assert rel <= 1e-6, f"norms: max rel error {rel:.3e} vs float64"


def _run_pair(run, rep, dtype):
    """(outputs for rep, outputs of the fp32 kernel for rep.float()); the same tuple twice for fp32 maps."""
    first = run(rep)
    second = run(rep.float()) if dtype == BF16 else first
    return first, second


@pytest.mark.parametrize("C,temp,kernels", REP_TEMP_CASES)
def test_rep_pass_model_temps(lib, C, temp, kernels):
    """The shipped fp32 student pass at the temperatures the models run it at."""
    import css_b200
    B, h, w = rep_shape("ragged")
    x, protos = rich_map(B, h, w, C, seed=3000 + 10 * C + int(1 / temp))
    prob, names = launched(lambda: css_b200.ops.proto_softmax_sim(x, protos, temp))
    assert_launched(kernels, names)
    check_sim_map(prob, x, protos, temp, "rep_pass")


# ---------------------------------------------------------------------------------------------------------------------------
# fused up-sample + softmax + max + fusion (css_sim.cu upsample_label_fuse_kernel)
# ---------------------------------------------------------------------------------------------------------------------------
def k2_smem(C, h, w, H, W):
    """Dynamic shared memory css_upsample_label_fuse asks for (css_sim.cu:618-626)."""
    ry = np.float32(h - 1) / np.float32(H - 1) if H > 1 else np.float32(0)
    rx = np.float32(w - 1) / np.float32(W - 1) if W > 1 else np.float32(0)
    in_th = int(min(h, math.ceil(ry * 7) + 3))
    in_tw = int(min(w, math.ceil(rx * 31) + 3))
    cp = (C + 3) & ~3 if C in (19, 21) else 32
    return 2 * cp * in_th * in_tw * 4


@pytest.mark.parametrize("C,h,w,H,W,temp,tile,kernel", UPSAMPLE_CASES)
def test_upsample_label_fuse(C, h, w, H, W, temp, tile, kernel):
    import css_b200
    from oracle import f64_ref as R
    smem = k2_smem(C, h, w, H, W)
    assert tile == ("global" if smem > 96 * 1024 else "optin" if smem > 48 * 1024 else "staged"), (tile, smem)
    g = torch.Generator().manual_seed(C * 7 + h)
    B = 2
    sim = (2 * torch.rand(B, C, h, w, generator=g) - 1).cuda()
    logits = (2.5 * torch.randn(B, C, h, w, generator=g)).cuda()
    o, names = launched(lambda: css_b200.ops.upsample_label_fuse(sim, logits, temp, (H, W), fuse="mix"))
    assert_launched([kernel], names)
    for key, src, t in (("rep", sim, temp), ("cls", logits, None)):
        conf, label, margin = R.upsample_softmax_max(src, (H, W), t)
        err = (o["conf_" + key].double() - conf).abs().max().item()
        bound = 2e-6
        if t in MODEL_TEMPS:
            f32 = torch.softmax(F.interpolate(src, size=(H, W), mode="bilinear", align_corners=True) / t, dim=1).max(dim=1).values
            bound = f32_bound(bound, (f32.double() - conf).abs().max().item(), f"torch float32 upsample conf t{t}")
        record(f"upsample conf t{t}" if t in MODEL_TEMPS else "upsample conf", err)
        assert err <= bound, f"conf_{key}: max abs error {err:.3e} vs float64 (bound {bound:.3e})"
        bad = o["label_" + key] != label
        assert not (bad & (margin >= TAU)).any(), f"label_{key} differs away from near-ties"
    fused = torch.where(o["label_rep"] == o["label_cls"], o["label_cls"].float(), torch.full_like(o["fused"], 255.0))
    assert torch.equal(o["fused"], fused)


# ---------------------------------------------------------------------------------------------------------------------------
# scorer (css_score.cu): gradient / no gradient x fixed-reference / online softmax x fp32 paths / bf16 x drawn / fed
# ---------------------------------------------------------------------------------------------------------------------------
def scorer_inputs(B2, C, h, w, seed, dtype=torch.float32):
    from css_b200 import synth
    d = synth.student_batch(B2, C, h, w, seed=seed, block=3 if h < 40 else 8)
    rep = d["rep"].to(dtype).cuda()
    protos = synth.warm_prototypes(C, seed=seed + 1, zero_rows=(1,)).cuda()
    return rep, d["label"].cuda(), d["mask"].cuda(), d["prob"].cuda(), protos


def run_loss(lib, variant, rep, label, mask, prob, protos, kw, seed, draws="fly", indices=None):
    """One Contrast_Loss call (forward, and backward for the gradient variants) on a fresh module; returns
    (loss, grad or None, module, the prototypes before the call, indices used)."""
    import css_b200
    lib.css_set_scorer_path(SCORER_PATH.get(variant, -1))
    crit = css_b200.Contrast_Loss(seed=seed, **kw).cuda()
    p0 = protos.clone()
    p = protos.clone()
    if variant.startswith("grad"):
        r = rep.detach().clone().requires_grad_(True)
        loss = crit(r, label, mask, prob, p, _indices=indices)
        loss.backward()
        return loss, r.grad, crit, p0, p
    with torch.no_grad():
        loss = crit(rep, label, mask, prob, p, _indices=indices)
    return loss, None, crit, p0, p


def f64_of(crit, rep, label, mask, p0, a, n, kw):
    from oracle import f64_ref as R
    return R.contrast_loss(rep, label, mask, p0, crit.selection(), a, n, temp=kw["temp"], alpha=kw["alpha"])


def check_against_f64(variant, loss, grad, crit, p0, p, rep, label, mask, kw, a, n, family):
    l64, g64, p64 = f64_of(crit, rep, label, mask, p0, a, n, kw)
    check_loss(loss, l64, family=family)
    torch.testing.assert_close(p.double(), p64, rtol=RTOL, atol=1e-6)
    if grad is not None:
        if grad.dtype == torch.bfloat16:
            # the gradient of a bf16 map is returned in bf16 (torch's convention): one bf16 rounding, rel 2^-8 at most
            check_grad(grad, g64, rtol=2 ** -8, family=family + " bf16")
        else:
            check_grad(grad, g64, family=family)


@pytest.mark.parametrize("variant,temp,draws,kernels", SCORER_CASES)
def test_scorer(lib, variant, temp, draws, kernels):
    B2, C, h, w, Q, Nn, seed = 2, 7, 19, 23, 12, 100, 31
    dt = torch.bfloat16 if variant.endswith("bf16") else torch.float32
    rep, label, mask, prob, protos = scorer_inputs(B2, C, h, w, seed, dt)
    kw = dict(num_queries=Q, num_negatives=Nn, temp=temp, strong_threshold=0.97, alpha=0.99)
    indices = None
    if draws == "fed":                        # the draws the on-the-fly sampler makes, materialised and fed back
        _, _, c0, _, _ = run_loss(lib, "nograd-f32", rep, label, mask, prob, protos, kw, seed)
        indices = c0.sample_indices(seed, 0)

    def both():
        first = run_loss(lib, variant, rep, label, mask, prob, protos, kw, seed, indices=indices)
        ref = run_loss(lib, "grad-f32-reg", rep.float(), label, mask, prob, protos, kw, seed) if variant.startswith("nograd") else None
        return first, ref
    ((loss, grad, crit, p0, p), ref), names = launched(both)
    assert_launched(kernels, names)
    a, n = indices if indices is not None else crit.sample_indices(seed, 0)
    check_against_f64(variant, loss, grad, crit, p0, p, rep, label, mask, kw, a, n, "scorer")
    if ref is not None:                       # same draws, same rows: the forward-only kernel agrees with the gradient kernel
        l_grad = ref[0]
        err = abs(loss.item() - l_grad.item()) / abs(l_grad.item())
        record(f"scorer no-grad vs path-0 loss (rel, {'bf16' if dt == torch.bfloat16 else 'f32'})", err)
        MAX_ERR.setdefault("scorer no-grad loss bit-identical to path 0", True)
        if loss.item() != l_grad.item():
            MAX_ERR["scorer no-grad loss bit-identical to path 0"] = False
        assert err <= 1e-6


@pytest.mark.parametrize("variant,Nn,kernels", NN_EDGE_CASES)
def test_scorer_candidate_counts(lib, variant, Nn, kernels):
    """Nn around the 32-candidate batch of a warp and a single negative."""
    B2, C, h, w, Q, seed = 2, 5, 13, 15, 9, 5 + Nn
    rep, label, mask, prob, protos = scorer_inputs(B2, C, h, w, seed)
    kw = dict(num_queries=Q, num_negatives=Nn, temp=0.5, strong_threshold=0.97, alpha=0.99)
    (loss, grad, crit, p0, p), names = launched(lambda: run_loss(lib, variant, rep, label, mask, prob, protos, kw, seed))
    assert_launched(kernels, names)
    a, n = crit.sample_indices(seed, 0)
    check_against_f64(variant, loss, grad, crit, p0, p, rep, label, mask, kw, a, n, "scorer")


@pytest.mark.parametrize("temp,kernels", TEMP_SWITCH_CASES)
def test_scorer_temperature_switch(lib, temp, kernels):
    """0.0240 takes the online-max softmax, 0.0241 the fixed reference (css_score.cu:863)."""
    B2, C, h, w, Q, Nn, seed = 2, 6, 17, 16, 10, 70, 77
    rep, label, mask, prob, protos = scorer_inputs(B2, C, h, w, seed)
    kw = dict(num_queries=Q, num_negatives=Nn, temp=temp, strong_threshold=0.97, alpha=0.99)

    def both():
        return (run_loss(lib, "grad-f32-reg", rep, label, mask, prob, protos, kw, seed),
                run_loss(lib, "nograd-f32", rep, label, mask, prob, protos, kw, seed))
    ((loss, grad, crit, p0, p), (l_ng, _, _, _, _)), names = launched(both)
    assert_launched(kernels, names)
    a, n = crit.sample_indices(seed, 0)
    check_against_f64("grad-f32-reg", loss, grad, crit, p0, p, rep, label, mask, kw, a, n, "scorer")
    assert abs(l_ng.item() - loss.item()) <= 1e-6 * abs(loss.item())


@pytest.mark.parametrize("temp", [0.0240, 0.0241])
def test_scorer_anti_aligned_candidates(lib, temp):
    """Every candidate, the positive included, nearly anti-aligned with every anchor: z - m is about -119 for all of them, so
    the fixed-reference weights 2^(z - m) sit near the bottom of the fp32 range (they must not flush to zero)."""
    B2, C, h, w, Q, Nn, seed = 1, 2, 12, 14, 8, 40, 3
    g = torch.Generator().manual_seed(seed)
    u = torch.randn(256, generator=g)
    u = 16 * u / u.norm()
    cls = (torch.arange(h * w) % 2).reshape(1, h, w)
    sign = (1 - 2 * cls).float()                                     # class 0: +u, class 1: -u
    rep = (sign[:, None] * u[None, :, None, None] + 0.15 * torch.randn(B2, 256, h, w, generator=g))
    label = torch.nn.functional.one_hot(cls, C).permute(0, 3, 1, 2).float()
    mask = torch.ones(B2, 1, h, w)
    prob = torch.full((B2, C, h, w), 0.5)                            # every valid pixel is hard
    protos = torch.stack([-u, u])                                    # each class's positive points the other way
    rep, label, mask, prob, protos = (t.cuda() for t in (rep, label, mask, prob, protos))
    kw = dict(num_queries=Q, num_negatives=Nn, temp=temp, strong_threshold=0.97, alpha=0.99)
    (loss, grad, crit, p0, p), names = launched(lambda: run_loss(lib, "grad-f32-reg", rep, label, mask, prob, protos, kw, seed))
    assert_launched([scorer_kernel("grad-f32-reg", temp > FIX_SWITCH, False)], names)
    a, n = crit.sample_indices(seed, 0)
    l64, g64, _ = f64_of(crit, rep, label, mask, p0, a, n, kw)
    assert l64 > 1.0                                                 # all logits are close: the loss is about log(Nn + 1)
    check_loss(loss, l64, family="scorer anti-aligned")
    check_grad(grad, g64, family="scorer anti-aligned")


def test_scorer_zero_norm_negative(lib):
    """A zero pixel among the valid (not hard) pixels, fed as a negative of every query: its norm is clamped at 1e-8 as
    torch.cosine_similarity does since 1.12, so its cosine is exactly 0 (no NaN)."""
    B2, C, h, w, Q, Nn, seed = 2, 4, 15, 17, 6, 20, 9
    rep, label, mask, prob, protos = scorer_inputs(B2, C, h, w, seed)
    cls = label.argmax(1)
    ys, xs = torch.nonzero((mask[0, 0] > 0) & (label[0].sum(0) > 0), as_tuple=True)
    y, x = int(ys[0]), int(xs[0])
    zc = int(cls[0, y, x])
    rep[0, :, y, x] = 0
    prob[0, zc, y, x] = 1.0                                           # valid but not hard: never an anchor
    kw = dict(num_queries=Q, num_negatives=Nn, temp=0.5, strong_threshold=0.97, alpha=0.99)
    _, _, c0, _, _ = run_loss(lib, "nograd-f32", rep, label, mask, prob, protos, kw, seed)
    sel = c0.selection()
    a, n = c0.sample_indices(seed, 0)
    px = y * w + x
    kz = sel["present"].index(zc)
    V = sel["V"]
    for k in range(V):
        if k == kz or sel["n_hard"][k] == 0:
            continue
        order = [(k + 1 + i) % V for i in range(V - 1)]              # rotated slots k+1..V-1, 0..k-1 (loss.py:139,141)
        off = sum(sel["num_list"][s] for s in order[:order.index(kz)])
        n[k, :, 0] = off + int(np.flatnonzero(sel["valid_ids"][kz] == px)[0])
    for variant in ("grad-f32-reg", "grad-f32-ring", "grad-f32-bulk", "nograd-f32"):
        loss, grad, crit, p0, p = run_loss(lib, variant, rep, label, mask, prob, protos, kw, seed, indices=(a, n))
        assert torch.isfinite(loss)
        check_against_f64(variant, loss, grad, crit, p0, p, rep, label, mask, kw, a, n, "scorer zero-norm")


@pytest.mark.parametrize("B2,C,h,w,kernels", BENCH_CASES)
def test_scorer_bench_shapes(lib, B2, C, h, w, kernels):
    """The shapes bench.py times: Q=256, Nn=512 on VOC 81x81 (B2=16) and CityScapes 193x193 (B2=8)."""
    Q, Nn, seed = 256, 512, 2024 + C
    rep, label, mask, prob, protos = scorer_inputs(B2, C, h, w, seed)
    kw = dict(num_queries=Q, num_negatives=Nn, temp=0.5, strong_threshold=0.97, alpha=0.99)
    (loss, grad, crit, p0, p), names = launched(lambda: run_loss(lib, "grad-f32-bulk", rep, label, mask, prob, protos, kw, seed))
    assert_launched(kernels, names)
    a, n = crit.sample_indices(seed, 0)
    check_against_f64("grad-f32-bulk", loss, grad, crit, p0, p, rep, label, mask, kw, a, n, "scorer bench")


# ---------------------------------------------------------------------------------------------------------------------------
# rows_verify_kernel<bf16>: DistributedDataParallel's clone of a bf16 rep_all
# ---------------------------------------------------------------------------------------------------------------------------
def test_rows_verify_bf16(lib):
    import css_b200
    from css_b200 import _lib
    B2, C, h, w = 2, 7, 24, 20
    rep, label, mask, _, protos = scorer_inputs(B2, C, h, w, 2, torch.bfloat16)
    kw = dict(num_queries=8, num_negatives=16, temp=0.5, strong_threshold=0.8, seed=4)

    def run(rep_in, prob):
        crit = css_b200.Contrast_Loss(**kw).cuda()
        with torch.no_grad():
            loss = crit(rep_in, label, mask, prob, protos.clone())
        return loss.item(), crit.last

    base, last = run(rep, css_b200.ops.proto_softmax_sim(rep, protos, 0.5))
    assert last["rows_cache_mode"] == "same"
    prob = css_b200.ops.proto_softmax_sim(rep, protos, 0.5)
    (l_clone, last), names = launched(lambda: run(rep.clone(), prob))
    assert_launched(ROWS_VERIFY_KERNELS, names)
    assert last["rows_cache_mode"] == "verify" and l_clone == base
    assert int(last["ws"].meta[_lib.META_ROWS_STALE].item()) == 0
    # one sampled channel changed (pixel 0 is checked on channels 0..3 by the first lanes of warp 0): flag raised, rows refreshed
    hit = torch.zeros_like(rep, dtype=torch.bool)
    hit[0, 0, 0, 0] = True
    other = torch.where(hit, rep + 1, rep)                          # out of place: a fresh tensor at version 0, as DDP's clone
    prob = css_b200.ops.proto_softmax_sim(rep, protos, 0.5)
    l_other, last = run(other, prob)
    assert last["rows_cache_mode"] == "verify"
    assert int(last["ws"].meta[_lib.META_ROWS_STALE].item()) == 1
    assert torch.equal(last["rows"], other.permute(0, 2, 3, 1).reshape(-1, 256))
    l_ref, last_ref = run(other, prob.clone())
    assert last_ref["rows_cache_mode"] == "miss" and l_other == l_ref


# ---------------------------------------------------------------------------------------------------------------------------
# channels-last maps (css_sim_tc.cu rep_pass_nhwc_kernel, rows_verify_rm_kernel; css_grad.cu grad_rows_kernel)
# ---------------------------------------------------------------------------------------------------------------------------
def nhwc_shape(shape):
    if shape == "one_tile":
        return 1, 9, 11                       # N = 99: one partial tile, rows past N zero-filled by the TMA
    if shape == "exact128":
        return 4, 8, 12                       # N = 384 = 3 x 128, tiles straddle image boundaries (h*w = 96)
    if shape == "ragged":
        return 3, 17, 29                      # N = 1479: partial last tile, straddling tiles
    if shape == "sub_wave":                   # one tile per CTA on all but a couple of SMs
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        h, w = 96, (sms - 2) * 128 // (2 * 96)
        assert math.ceil(2 * h * w / 128) < sms
        return 2, h, w
    return 8, 193, 193                        # city193: ~16 tiles per CTA, every ring and both TMEM buffers wrap their parity


def to_channels_last(x):
    return x.contiguous(memory_format=torch.channels_last)


@pytest.mark.parametrize("C,shape,temp,kernels", NHWC_CASES)
def test_nhwc_rep_pass(lib, C, shape, temp, kernels):
    """ops.cos_sim_map / proto_softmax_sim on a torch.channels_last map, on both sides of the C <= 24 switch (C 25..31 leave
    padded class columns in the accumulators, which must not reach a softmax)."""
    import css_b200
    B, h, w = nhwc_shape(shape)
    x, protos = rich_map(B, h, w, C, seed=5000 + 100 * C + h)
    rep = to_channels_last(x)
    assert css_b200.ops.is_channels_last(rep)
    if temp is None:
        out, names = launched(lambda: css_b200.ops.cos_sim_map(rep, protos))
    else:
        out, names = launched(lambda: css_b200.ops.proto_softmax_sim(rep, protos, temp))
    assert_launched(kernels, names)
    check_sim_map(out, rep, protos, temp, "nhwc")
    if temp is not None:
        cache = out._css_rows
        assert cache.rows.data_ptr() == rep.data_ptr()                  # the map is its own row table
        check_norms(cache.norms, rep, "nhwc")


@pytest.mark.parametrize("offset,kernels", NHWC_ALIGN_CASES)
def test_nhwc_alignment(lib, offset, kernels):
    """A channels-last map at 4 floats into a buffer (16-byte, not 1 KB aligned) is read by the TMA kernel as it is; at 1 float
    is_channels_last refuses it and the pass runs on the contiguous NCHW copy."""
    import css_b200
    B, C, h, w = 2, 21, 13, 11
    x, protos = rich_map(B, h, w, C, seed=77 + offset)
    buf = torch.full((x.numel() + 4,), float("nan"), device="cuda")
    rep = buf.as_strided(x.shape, (h * w * 256, 1, w * 256, 256), offset)
    rep.copy_(x)
    assert rep.data_ptr() % 16 == 4 * offset % 16 and rep.data_ptr() % 1024 != 0
    assert css_b200.ops.is_channels_last(rep) == (offset == 4)
    prob, names = launched(lambda: css_b200.ops.proto_softmax_sim(rep, protos, 0.5))
    assert_launched(kernels, names)
    if offset != 4:
        assert not {n for n in names if n.startswith("rep_pass_nhwc_kernel")}
    check_sim_map(prob, x, protos, 0.5, "nhwc")
    rows = prob._css_rows.rows
    assert torch.equal(rows, x.permute(0, 2, 3, 1).reshape(-1, 256))
    assert (rows.data_ptr() == rep.data_ptr()) == (offset == 4)
    check_norms(prob._css_rows.norms, x, "nhwc")


def test_nhwc_norms_and_rows_check(lib):
    """The norms-only pass (css_rep_pass_nhwc without prototypes) and css_rows_refresh_nhwc: an intact clone leaves the flag at 0
    and the norms untouched (the pass returns at its guard); a clone that differs in one sampled channel of the last pixel,
    ((p * 37) & 63) + 64 i (css_sim_tc.cu rows_verify_rm_kernel), raises the flag and has its norms rewritten."""
    import css_b200
    from css_b200 import _lib
    from css_b200._lib import check, ptr, stream_ptr
    B, h, w = 3, 17, 29
    N = B * h * w
    x, _ = rich_map(B, h, w, 1, seed=91)
    rep = to_channels_last(x)
    norms, names = launched(lambda: css_b200.ops.rep_norms_nhwc(rep))
    assert_launched([nhwc_kernel(1)], names)
    check_norms(norms, x, "nhwc")
    scratch = torch.empty(2 * 256 * 32, device="cuda")

    def refresh(clone, out):
        meta = torch.zeros(_lib.META_WORDS, device="cuda", dtype=torch.int32)
        check(lib.css_rows_refresh_nhwc(ptr(clone), ptr(rep), ptr(out), ptr(scratch), ptr(meta), B, 256, h, w, stream_ptr()),
              "css_rows_refresh_nhwc")
        return int(meta[_lib.META_ROWS_STALE].item())

    clone = rep.clone()
    assert clone.stride() == rep.stride() and clone.data_ptr() != rep.data_ptr()
    sentinel = torch.full((N,), -7.0, device="cuda")
    flag, names = launched(lambda: refresh(clone, sentinel))
    assert_launched(NHWC_REFRESH_KERNELS, names)
    assert flag == 0 and (sentinel == -7.0).all()
    p = N - 1
    for i in range(4):
        other = rep.clone()
        css_b200.ops.rows_view(other)[p, ((p * 37) & 63) + 64 * i] += 0.5
        out = torch.full((N,), -7.0, device="cuda")
        assert refresh(other, out) == 1, f"a change in sampled channel {((p * 37) & 63) + 64 * i} of pixel {p} went unnoticed"
        check_norms(out, other, "nhwc")


def grad_anchors(spread, N, n, rng):
    if spread == "uniform":
        return rng.integers(0, N, n)
    if spread == "dups":                      # seven distinct pixels hit ~150 times each, 30 % of the slots without an anchor
        px = rng.choice(rng.integers(0, N, 7), n)
        px[rng.random(n) < 0.3] = -1
        return px
    px = rng.integers(0, N, n)                # "hot": the last pixel hit 600 times among uniform anchors
    px[rng.choice(n, 600, replace=False)] = N - 1
    return px


GRAD_NHWC_CASES = {"dups_and_absent": (3, 10, 12, 1501, "dups"), "hot_pixel": (2, 21, 23, 2005, "hot"),
                   "uniform": (4, 81, 81, 2003, "uniform"), "over_32k_anchors": (2, 16, 16, 33003, "uniform")}


@pytest.mark.parametrize("name", list(GRAD_NHWC_CASES))
def test_nhwc_grad_scatter(lib, name):
    """css_grad_scatter_nhwc against a float64 scatter-add.  n_anchor is never a multiple of the 8 anchors of a CTA.  The output
    is NaN-filled with guard elements on both sides that must stay NaN.  fp32 atomics add in any order: an element with k
    contributions t_i is bounded by gamma_(k+1) sum |t_i|, gamma_m = m u / (1 - m u), u = 2^-24 (one rounding per product)."""
    from css_b200._lib import check, ptr, stream_ptr
    B2, h, w, n, spread = GRAD_NHWC_CASES[name]
    N = B2 * h * w
    rng = np.random.default_rng(n)
    px = torch.from_numpy(grad_anchors(spread, N, n, rng).astype(np.int32)).cuda()
    ga = torch.from_numpy(rng.standard_normal((n, 256)).astype(np.float32)).cuda()
    go = torch.full((), 0.37, device="cuda")
    G = 4
    buf = torch.full((N * 256 + 2 * G,), float("nan"), device="cuda")
    out = buf[G:G + N * 256]

    def run():
        check(lib.css_grad_scatter_nhwc(ptr(go), ptr(px), ptr(ga), n, B2, 256, h, w, ptr(out), stream_ptr()), "css_grad_scatter_nhwc")
    _, names = launched(run)
    assert_launched(["grad_rows_kernel"], names)
    assert torch.isnan(buf[:G]).all() and torch.isnan(buf[G + N * 256:]).all(), "written outside the gradient"
    keep = px >= 0
    terms = go.double() * ga[keep].double()
    ref = torch.zeros(N, 256, dtype=torch.float64, device="cuda").index_add_(0, px[keep].long(), terms)
    mag = torch.zeros_like(ref).index_add_(0, px[keep].long(), terms.abs())
    k = torch.bincount(px[keep].long(), minlength=N).double()[:, None] + 1
    u = 2.0 ** -24
    bound = k * u / (1 - k * u) * mag
    got = out.view(N, 256).double()
    assert torch.isfinite(got).all()
    assert torch.equal(got != 0, ref != 0), "the gradient's support is not the anchor pixels"
    err = (got - ref).abs()
    record("nhwc grad scatter: max |err| / rigorous bound", (err / bound.clamp_min(1e-300)).max())
    assert (err <= bound).all(), f"max excess {(err - bound).max().item():.3e}"
    if spread == "hot":
        assert int(k[N - 1]) > 600


@pytest.mark.parametrize("temp", [0.5, 0.02])
def test_nhwc_contrast_loss(lib, temp):
    """Contrast_Loss on a channels-last map handed over as DDP's clone (rows check on the device), with fed draws: loss,
    gradient and prototypes against float64; the gradient keeps the map's channels-last strides."""
    import css_b200
    B2, C, h, w, Q, Nn, seed = 2, 7, 19, 23, 12, 100, 31
    rep0, label, mask, _, protos = scorer_inputs(B2, C, h, w, seed)
    rep0 = to_channels_last(rep0)
    prob = css_b200.ops.proto_softmax_sim(rep0, protos, 0.5)
    kw = dict(num_queries=Q, num_negatives=Nn, temp=temp, strong_threshold=0.8, alpha=0.99)
    _, _, c0, _, _ = run_loss(lib, "nograd-f32", rep0, label, mask, prob, protos, kw, seed)
    a, n = c0.sample_indices(seed, 0)

    def step():
        rep = rep0.clone().requires_grad_(True)
        crit = css_b200.Contrast_Loss(seed=seed, **kw).cuda()
        p = protos.clone()
        loss = crit(rep, label, mask, prob, p, _indices=(a, n))
        loss.backward()
        return loss, rep, crit, p
    (loss, rep, crit, p), names = launched(step)
    assert_launched(NHWC_LOSS_KERNELS, names)
    assert crit.last["rows_cache_mode"] == "verify"
    assert int(crit.last["ws"].meta[css_b200._lib.META_ROWS_STALE].item()) == 0
    assert rep.grad.stride() == rep0.stride()
    check_against_f64("grad-f32", loss, rep.grad, crit, protos, p, rep0, label, mask, kw, a, n, "nhwc")


# ---------------------------------------------------------------------------------------------------------------------------
# NCHW tensor-core rep pass (css_sim_tc.cu rep_pass_tc_kernel<ROWS, NP>, proto_prep_tc_kernel)
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def tc_lib():
    from css_b200 import _lib
    lib = _lib.load()
    lib.css_set_rep_pass_path(1)
    yield lib
    lib.css_set_rep_pass_path(-1)


@pytest.mark.parametrize("C,shape,offset,temp,kernels", TC_CASES)
def test_tc_rep_pass(tc_lib, C, shape, offset, temp, kernels):
    """Cosine map, or softmax + rows + norms, with the map `offset` floats into its buffer."""
    import css_b200
    B, h, w = TC_SHAPES[shape]
    x, protos = rich_map(B, h, w, C, seed=7000 + 100 * C + 10 * offset + h)
    buf = torch.full((x.numel() + 4,), float("nan"), device="cuda")
    rep = buf[offset:offset + x.numel()].view(x.shape)
    rep.copy_(x)
    assert rep.data_ptr() % 16 == 4 * offset
    if temp is None:
        out, names = launched(lambda: css_b200.ops.cos_sim_map(rep, protos))
    else:
        out, names = launched(lambda: css_b200.ops.proto_softmax_sim(rep, protos, temp))
    assert_launched(kernels, names)
    check_sim_map(out, x, protos, temp, "tc")
    if temp is not None:
        assert torch.equal(out._css_rows.rows, x.permute(0, 2, 3, 1).reshape(-1, 256))
        check_norms(out._css_rows.norms, x, "tc")


# ---------------------------------------------------------------------------------------------------------------------------
# Attention_Threshold_Loss, generic class count (css_atl.cu <0> kernels; the finaliser walks images 8 at a time)
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,B,kernels", ATL_CASES)
def test_atl_generic(C, B, kernels):
    import css_b200
    from oracle import f64_ref as R
    H, W, thr = 11, 13, 0.8
    g = torch.Generator().manual_seed(C * 1000 + B)
    pred = 2.0 * torch.randn(B, C, H, W, generator=g)
    label = torch.randint(0, C, (B, H, W), generator=g)
    label = torch.where(torch.rand(B, H, W, generator=g) < 0.1, torch.full_like(label, -1), label)
    conf = torch.rand(B, H, W, generator=g)
    if B > 1:
        conf[B // 2] = 0.5 * conf[B // 2]                            # an image with no confident pixel (weighting 0)
        label[B - 1] = -1                                            # an all-ignored image (weighting 0/0, no selected pixel)
    pred, label, conf = pred.cuda().requires_grad_(True), label.cuda(), conf.cuda()
    crit = css_b200.Attention_Threshold_Loss(thr)

    def fwd_bwd():
        loss = crit(pred, label, conf)
        loss.backward()
        return loss
    loss, names = launched(fwd_bwd)
    assert_launched(kernels, names)
    l64, g64 = R.attention_threshold_loss(pred, label, conf, thr)
    check_loss(loss, l64, family="atl")
    check_grad(pred.grad, g64, family="atl")


# ---------------------------------------------------------------------------------------------------------------------------
# peer-memory exchange (css_comm.cu stats_allreduce_kernel<WMAX>): worlds 3, 5 and 9 as process groups of one 9-process job
# ---------------------------------------------------------------------------------------------------------------------------
def _peer_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(0)
    from css_b200 import _lib
    from css_b200.comm import PeerStatsReducer
    _lib.check(_lib.load().css_comm_set_timeout_ms(120_000), "css_comm_set_timeout_ms")
    C, D = 19, 256
    groups = {n: dist.new_group(list(range(n))) for n in PEER_WORLDS}     # collective: every rank creates every group
    res = {}
    for n in PEER_WORLDS:
        if rank >= n:
            continue

        def block(it, r):
            return torch.randn(C, D + 1, generator=torch.Generator().manual_seed(1000 * it + 37 * n + r))

        def expected(it):
            s = torch.zeros(C, D + 1)
            for r in range(n):                                       # rank order, as the kernel sums
                s = s + block(it, r)
            return s

        red = PeerStatsReducer("cuda:0", groups[n])
        r = dict(ok=red.ok, errs=[], graph_errs=[], sums=[])
        if red.ok:
            def epochs():
                for it in range(4):                                  # both slot parities
                    x = block(it, rank).cuda()
                    red.allreduce(x, C, D)
                    r["sums"].append(x.cpu())
            _, names = launched(epochs)
            r["launched"] = peer_kernel(n) in names
            r["errs"] = [float((s - expected(it)).abs().max()) for it, s in enumerate(r["sums"])]
            static = torch.zeros(C, D + 1).cuda()
            side = torch.cuda.Stream()
            with torch.cuda.stream(side):
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=side):
                    red.allreduce(static, C, D)
            for it in range(10, 12):
                static.copy_(block(it, rank))
                graph.replay()
                torch.cuda.synchronize()
                r["graph_errs"].append(float((static.cpu() - expected(it)).abs().max()))
                r["sums"].append(static.cpu())
            r["timeouts"] = red.timeouts()
            dist.barrier(group=groups[n])
            red.close()
        r["sums"] = [s.numpy() for s in r["sums"]]
        res[n] = r
    dist.barrier()
    out[rank] = res
    dist.destroy_process_group()


def test_peer_exchange_worlds():
    """Rank-ordered sums, bit-identical on every rank, over several epochs and CUDA-graph replays, with a bounded timeout."""
    import torch.multiprocessing as mp
    world = max(PEER_WORLDS)
    port = 29400 + (os.getpid() % 90)
    mgr = mp.Manager()
    try:
        out = mgr.dict()
        mp.spawn(_peer_worker, args=(world, port, out), nprocs=world, join=True)
        res = {r: out[r] for r in range(world)}
    finally:
        mgr.shutdown()
    for n in PEER_WORLDS:
        oks = {res[r][n]["ok"] for r in range(n)}
        assert len(oks) == 1
        if not oks.pop():
            pytest.skip("CUDA IPC between the test processes is not available on this box")
        for r in range(n):
            got = res[r][n]
            assert got["launched"], f"world {n} rank {r}: {peer_kernel(n)} not launched"
            assert got["timeouts"] == 0, (n, r, got["timeouts"])
            assert got["errs"] == [0.0] * 4 and got["graph_errs"] == [0.0] * 2, (n, r, got["errs"], got["graph_errs"])
            for a, b in zip(got["sums"], res[0][n]["sums"]):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
