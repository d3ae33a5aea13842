"""css_b200.install.install() against an unmodified reference checkout (WangChangqi98/CSS), named by $CSS_REFERENCE_ROOT;
without one this test skips.  Checks that the names the scripts import are replaced and that the shells are
wired to the reference's own network / augmentation functions."""
import os
import sys

import pytest

REF = os.environ.get("CSS_REFERENCE_ROOT", "")


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "generalframeworks")), reason="no reference checkout: set CSS_REFERENCE_ROOT")
def test_install_patches_reference_modules():
    import torch
    import torch.distributed as dist
    import css_b200
    from css_b200 import install, models
    saved_hooks = dict(vars(models.hooks))
    saved_mods = {k: v for k, v in sys.modules.items() if k.startswith("generalframeworks") or k == "shutup"}
    try:
        ref_model, ref_loss = install.install(reference_root=REF)
        assert ref_loss.Contrast_Loss is css_b200.Contrast_Loss
        assert ref_loss.Attention_Threshold_Loss is css_b200.Attention_Threshold_Loss
        assert ref_model.Model_mix is css_b200.Model_mix and ref_model.Model_cross is css_b200.Model_cross
        assert ref_model.Model_ori_pseudo is css_b200.Model_ori_pseudo
        assert "shutup" in sys.modules and callable(sys.modules["shutup"].please)
        assert models.hooks.network_factory is ref_model.DeepLabv3Plus_with_rep
        # same constructor surface as the scripts use (mix_label.py:75,83-87)
        crit = ref_loss.Contrast_Loss(strong_threshold=0.8, num_queries=256, num_negatives=512, temp=0.5, alpha=0.99)
        assert (crit.num_queries, crit.num_negatives, crit.temp, crit.strong_threshold, crit.alpha) == (256, 512, 0.5, 0.8, 0.99)
        import torchvision.models as tvm
        m = ref_model.Model_mix(tvm.resnet18(), num_classes=21, output_dim=256, config={"Dataset": {}}, temp=0.5)
        assert hasattr(m, "model") and hasattr(m, "ema_model") and m.step == 0 and m.temp == 0.5
        assert all(not p.requires_grad for p in m.ema_model.parameters())
        before = [p.detach().clone() for p in m.ema_model.parameters()]
        with torch.no_grad():
            for p in m.model.parameters():
                p.add_(1.0)
        m.ema_update()                      # step 0: decay = min(1 - 1/1, alpha) = 0 -> teacher := student (ddp_model.py:93-97)
        assert m.step == 1
        for e, s in zip(m.ema_model.parameters(), m.model.parameters()):
            assert torch.allclose(e, s)
        m.ema_update()                      # step 1: decay = 0.5
        assert m.step == 2 and len(before) > 0
        # gpu_aug=True points the augmentation hooks at css_b200.aug (maps stay on the GPU), the default at the reference
        from css_b200 import aug
        assert models.hooks.batch_transform_2 is not aug.batch_transform_2
        install.install(reference_root=REF, gpu_aug=True)
        assert models.hooks.batch_transform_2 is aug.batch_transform_2
        assert models.hooks.generate_cut_gather_3 is aug.generate_cut_gather_3
    finally:
        for k, v in saved_hooks.items():
            setattr(models.hooks, k, v)
        if dist.is_initialized() and not saved_mods:
            pass
