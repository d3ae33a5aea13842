"""Drops the CUDA path into an unmodified checkout of the reference (WangChangqi98/CSS).

    import css_b200.install; css_b200.install.install()      # BEFORE importing ori_pseudo / mix_label / cross_label

The three scripts bind their names with `from ... import` at import time (mix_label.py:12,21), so the reference modules
are patched first: `generalframeworks.loss.loss.Contrast_Loss` (and the two logit-space losses) and `generalframeworks.networks.ddp_model.Model_*` are
replaced by the css_b200 classes, whose hooks are pointed at the reference's own network and augmentation functions.
"""
import importlib
import sys
import types


def install(reference_root=None, stub_shutup=True, gpu_aug=False):
    """gpu_aug=True also routes the shells' augmentation calls through css_b200.aug: the label / confidence maps stay on the
    GPU (same outputs, same RNG consumption as dataset_helpers/VOC.py:312-477); the default keeps the reference's functions."""
    if reference_root and reference_root not in sys.path:
        sys.path.insert(0, reference_root)
    if stub_shutup and "shutup" not in sys.modules:
        try:
            importlib.import_module("shutup")
        except ImportError:                       # the scripts do `import shutup; shutup.please()` (mix_label.py:1-2)
            m = types.ModuleType("shutup")
            m.please = lambda: None
            sys.modules["shutup"] = m
    ref_model = importlib.import_module("generalframeworks.networks.ddp_model")
    ref_loss = importlib.import_module("generalframeworks.loss.loss")
    from . import loss as _loss
    from . import models as _models
    h = _models.hooks
    h.network_factory = ref_model.DeepLabv3Plus_with_rep
    for name in ("batch_transform", "batch_transform_2", "batch_transform_3", "generate_cut_gather",
                 "generate_cut_gather_2", "generate_cut_gather_3"):
        # resolved through the reference module at call time, exactly like ddp_model.py:6,121,127,132 does
        setattr(h, name, (lambda n: (lambda *a, **k: getattr(ref_model, n)(*a, **k)))(name))
    if gpu_aug:
        from . import aug as _aug
        for name in ("batch_transform", "batch_transform_2", "batch_transform_3", "generate_cut_gather",
                     "generate_cut_gather_2", "generate_cut_gather_3"):
            setattr(h, name, getattr(_aug, name))
    ref_loss.Contrast_Loss = _loss.Contrast_Loss
    ref_loss.Attention_Threshold_Loss = _loss.Attention_Threshold_Loss
    ref_loss.ProbOhemCrossEntropy2d = _loss.ProbOhemCrossEntropy2d
    ref_model.Model_ori_pseudo = _models.Model_ori_pseudo
    ref_model.Model_mix = _models.Model_mix
    ref_model.Model_cross = _models.Model_cross
    return ref_model, ref_loss
