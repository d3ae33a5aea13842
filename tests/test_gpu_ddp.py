"""Script-level integration under DistributedDataParallel (SURVEY.md 8(b) "who calls it"): the reference wraps Model_mix in
DistributedDataParallel(..., find_unused_parameters=True) (mix_label.py:76-77) and calls the loss from train()
(mix_label.py:154-197).  With find_unused_parameters DDP's output sink CLONES every output that requires grad, so the loss
receives rep_all at a different address than the one the student pass read; the one-read property of the path must survive
that (css_rows_refresh), and gradients must reach the network through DDP.

  * test_train_body_under_ddp_stub_network      -- always runs: the body of train() restated statement by statement around
                                                   a small convolutional stub (no reference needed on the GPU box);
  * test_unmodified_mix_label_train_under_ddp   -- runs when the reference travelled to the box in baseline/_ref (git-ignored
                                                   copy made by __graft_entry__.build()): imports the UNMODIFIED mix_label.py
                                                   after css_b200.install.install() and calls its own train().
"""
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("CSS_REFERENCE_ROOT") or os.path.join(ROOT, "baseline", "_ref")


@pytest.fixture(scope="module")
def world1():
    """Single-process NCCL group on cuda:0, as mp.spawn + local_dist_init give each rank of the scripts (world size 1)."""
    created = False
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", str(29400 + os.getpid() % 90))
        torch.cuda.set_device(0)
        dist.init_process_group("nccl", rank=0, world_size=1)
        created = True
    yield
    if created:
        dist.destroy_process_group()


class StubNet(nn.Module):
    """Stands in for DeepLabv3Plus_with_rep: image [B,3,H,W] -> (pred [B,C,h,w], rep [B,256,h,w]) at stride 4."""

    def __init__(self, base_encoder=None, num_classes=21, output_dim=256, dilate_scale=8):
        super().__init__()
        self.stem = nn.Conv2d(3, 16, 3, stride=4, padding=1)
        self.cls = nn.Conv2d(16, num_classes, 1)
        self.rep = nn.Conv2d(16, output_dim, 1)
        self.unused = nn.Linear(4, 4)            # never used in forward: what find_unused_parameters=True is for

    def forward(self, x):
        f = torch.relu(self.stem(x))
        return self.cls(f), self.rep(f)


def _passthrough_hooks(models):
    saved = dict(vars(models.hooks))
    models.hooks.network_factory = StubNet
    models.hooks.batch_transform_2 = lambda img, lab, c1, c2, **k: (img, torch.where(lab == 255, torch.full_like(lab, -1), lab).long(),
                                                                     torch.floor(c1 * 255) / 255, torch.floor(c2 * 255) / 255)
    models.hooks.generate_cut_gather_2 = lambda a, b, c, d, mode=None: (a, b, c, d)
    return saved


def test_train_body_under_ddp_stub_network(world1):
    import css_b200
    from css_b200 import models
    from torch.nn.parallel import DistributedDataParallel
    saved = _passthrough_hooks(models)
    try:
        B, C, H, W = 2, 21, 129, 129
        config = {"Dataset": {"crop_size": (H, W), "scale_size": (1.0, 1.0), "mix_mode": "none", "name": "VOC"}, "Network": {"num_class": C}}
        args = types.SimpleNamespace(weak_threshold=0.7, sche=True)
        torch.manual_seed(0)
        model = css_b200.Model_mix(None, num_classes=C, output_dim=256, config=config, temp=0.5).cuda()
        model = nn.SyncBatchNorm.convert_sync_batchnorm(model).cuda()                              # mix_label.py:76
        model = DistributedDataParallel(model, device_ids=[torch.cuda.current_device()], find_unused_parameters=True)   # :77
        criterion = {"ce_loss": nn.CrossEntropyLoss(ignore_index=-1).cuda(),
                     "unsup_loss": css_b200.Attention_Threshold_Loss(strong_threshold=0.97).cuda(),
                     "contrast_loss": css_b200.Contrast_Loss(strong_threshold=0.8, num_queries=64, num_negatives=128, temp=0.5, alpha=0.99).cuda()}
        prototypes = torch.zeros(C, 256).cuda()                                                    # :93
        optimizer = torch.optim.SGD(model.module.model.parameters(), lr=1e-2, momentum=0.9, nesterov=True)
        g = torch.Generator().manual_seed(1)
        w_before = model.module.model.rep.weight.detach().clone()
        for it in range(3):
            # ---- mix_label.py:161-193, statement by statement ----
            train_l_image = torch.randn(B, 3, H, W, generator=g).cuda()
            train_l_label = torch.randint(-1, C, (B, H, W), generator=g).cuda()
            train_u_image = torch.randn(B, 3, H, W, generator=g).cuda()
            pred_l_large, pred_u_large, train_u_aug_label, train_u_aug_logits_cls, train_u_aug_logits_rep, rep_all, pred_all = \
                model(train_l_image, train_u_image, prototypes)
            sup_loss = criterion["ce_loss"](pred_l_large, train_l_label)
            unsup_loss = criterion["unsup_loss"](pred_u_large, train_u_aug_label, train_u_aug_logits_cls)
            with torch.no_grad():
                train_u_aug_mask = train_u_aug_logits_cls.ge(args.weak_threshold).float()
                mask_all = torch.cat(((train_l_label.unsqueeze(1) >= 0).float(), train_u_aug_mask.unsqueeze(1)))
                mask_all = F.interpolate(mask_all, size=pred_all.shape[2:], mode="nearest")
                label_l = F.interpolate(_label_onehot(train_l_label, C), size=pred_all.shape[2:], mode="nearest")
                label_u = F.interpolate(_label_onehot_2(train_u_aug_label, C), size=pred_all.shape[2:], mode="nearest")
                label_u = label_u[:, 1:, :, :]
                label_all = torch.cat((label_l, label_u))
            # what DDP(find_unused_parameters=True) does to the outputs: rep_all is a clone, prob_all passes through
            inner_rep = pred_all._css_rows.src
            assert rep_all.data_ptr() != inner_rep.data_ptr() and torch.equal(rep_all, inner_rep)
            contrast_loss = criterion["contrast_loss"](rep_all, label_all, mask_all, pred_all, prototypes)
            last = criterion["contrast_loss"].last
            assert last["rows_from_cache"] is True and last["rows_cache_mode"] == "verify"
            assert int(last["ws"].meta[css_b200._lib.META_ROWS_STALE].item()) == 0      # the device check found the rows intact
            # ... and they are the rows of the tensor the loss was given
            want = rep_all.detach().permute(0, 2, 3, 1).reshape(-1, 256)
            assert torch.equal(last["rows"], want)
            total_loss = sup_loss + unsup_loss + contrast_loss * 1.0
            optimizer.zero_grad()
            total_loss.backward()
            optimizer.step()
            model.module.ema_update()
            assert torch.isfinite(total_loss).item()
        assert not torch.equal(w_before, model.module.model.rep.weight)        # the contrastive gradient reached the network through DDP
        assert prototypes.abs().sum().item() > 0 and torch.isfinite(prototypes).all().item()
        assert model.module.step == 3
    finally:
        for k, v in saved.items():
            setattr(models.hooks, k, v)


def test_rows_cache_never_serves_stale_rows(world1):
    """The carried rows are used only when they ARE the rows of `rep`: a tensor with other content (fresh, version 0) makes
    the device check fail and the rows-only pass rewrite them; a tensor modified in place is not trusted at all."""
    import css_b200
    from css_b200 import synth
    B2, C, h, w = 2, 7, 24, 20
    d = synth.student_batch(B2, C, h, w, seed=2, strategy="mix", block=4)
    protos = synth.warm_prototypes(C, seed=3).cuda()
    rep = d["rep"].cuda()
    label, mask = d["label"].cuda(), d["mask"].cuda()
    kw = dict(num_queries=8, num_negatives=16, temp=0.5, strong_threshold=0.8, seed=4)

    def run(rep_in, prob, p):
        crit = css_b200.Contrast_Loss(**kw).cuda()
        loss = crit(rep_in, label, mask, prob, p)
        return loss.item(), crit.last

    prob = css_b200.ops.proto_softmax_sim(rep, protos, 0.5)
    base, last = run(rep, prob, protos.clone())
    assert last["rows_cache_mode"] == "same"
    # (a) a clone: verified on the device, same result bit for bit
    prob = css_b200.ops.proto_softmax_sim(rep, protos, 0.5)
    l_clone, last = run(rep.clone(), prob, protos.clone())
    assert last["rows_cache_mode"] == "verify" and l_clone == base
    assert int(last["ws"].meta[css_b200._lib.META_ROWS_STALE].item()) == 0
    # (b) different content under a fresh tensor: the check fails on the device, the rows are rewritten from the new tensor
    other = (rep * 1.5 + 0.25).contiguous()
    prob = css_b200.ops.proto_softmax_sim(rep, protos, 0.5)
    l_other, last = run(other, prob, protos.clone())
    assert last["rows_cache_mode"] == "verify"
    assert int(last["ws"].meta[css_b200._lib.META_ROWS_STALE].item()) == 1
    assert torch.equal(last["rows"], other.permute(0, 2, 3, 1).reshape(-1, 256))
    l_ref, last_ref = run(other, prob.clone(), protos.clone())          # prob.clone() carries nothing: the plain rows-only pass
    assert last_ref["rows_cache_mode"] == "miss" and l_other == l_ref
    # (c) a single pixel edited out of place (e.g. torch.where): caught, every pixel is sampled
    one2 = torch.where(_pixel_mask(rep, 1, 3, 5), torch.zeros_like(rep), rep)
    prob = css_b200.ops.proto_softmax_sim(rep, protos, 0.5)
    _, last = run(one2, prob, protos.clone())
    assert int(last["ws"].meta[css_b200._lib.META_ROWS_STALE].item()) == 1
    assert torch.equal(last["rows"], one2.permute(0, 2, 3, 1).reshape(-1, 256))
    # (d) modified in place after the student pass: version counter differs -> not trusted, plain rows-only pass
    prob = css_b200.ops.proto_softmax_sim(rep, protos, 0.5)
    rep.mul_(2.0)
    _, last = run(rep, prob, protos.clone())
    assert last["rows_cache_mode"] == "miss"
    assert torch.equal(last["rows"], rep.permute(0, 2, 3, 1).reshape(-1, 256))


def _pixel_mask(rep, b, y, x):
    m = torch.zeros_like(rep, dtype=torch.bool)
    m[b, :, y, x] = True
    return m


def _label_onehot(inputs, num_class):                       # generalframeworks/utils.py:116-125
    batch_size, image_h, image_w = inputs.shape
    inputs = torch.relu(inputs)
    outputs = torch.zeros([batch_size, num_class, image_h, image_w]).to(inputs.device)
    return outputs.scatter_(1, inputs.unsqueeze(1), 1.0)


def _label_onehot_2(inputs, num_class):                     # generalframeworks/utils.py:127-136
    batch_size, image_h, image_w = inputs.shape
    inputs = inputs + 1
    outputs = torch.zeros([batch_size, (num_class + 1), image_h, image_w]).to(inputs.device)
    return outputs.scatter_(1, inputs.unsqueeze(1), 1.0)


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "generalframeworks")) or not os.path.exists(os.path.join(REF, "mix_label.py")),
                    reason="no reference checkout in baseline/_ref or at CSS_REFERENCE_ROOT")
def test_unmodified_mix_label_train_under_ddp(world1):
    """The reference's OWN train() (mix_label.py:154-197, imported unmodified) driving the css_b200 classes that install()
    swapped in, with the reference's DeepLabv3+ (torchvision ResNet-50 trunk to keep the test light), its PIL augmentation and
    CutMix, under DistributedDataParallel(find_unused_parameters=True)."""
    import css_b200
    import css_b200.install
    import torchvision.models as tvm
    from torch.nn.parallel import DistributedDataParallel
    from torch.utils.data import DataLoader, TensorDataset
    from torch.utils.data.distributed import DistributedSampler
    css_b200.install.install(reference_root=REF)
    sys.modules.pop("mix_label", None)
    import mix_label                                           # the unmodified script (its __main__ block does not run)
    assert mix_label.Contrast_Loss is css_b200.Contrast_Loss and mix_label.Model_mix is css_b200.Model_mix
    from generalframeworks.scheduler.my_lr_scheduler import PolyLR
    from generalframeworks.scheduler.rampscheduler import RampdownScheduler
    B, C, H, W, iters = 2, 21, 161, 161, 2
    config = {"Dataset": {"name": "VOC", "crop_size": (H, W), "scale_size": (0.5, 1.5), "mix_mode": "cutmix", "batch_size": B},
              "Network": {"num_class": C}}
    args = types.SimpleNamespace(weak_threshold=0.7, sche=True, temp=0.5)
    torch.manual_seed(3407)
    np.random.seed(3407)
    model = mix_label.Model_mix(tvm.resnet50(), num_classes=C, output_dim=256, config=config, temp=args.temp).cuda()
    model = nn.SyncBatchNorm.convert_sync_batchnorm(model).cuda()
    model = DistributedDataParallel(model, device_ids=[torch.cuda.current_device()], find_unused_parameters=True)
    criterion = {"ce_loss": nn.CrossEntropyLoss(ignore_index=-1).cuda(),
                 "unsup_loss": mix_label.Attention_Threshold_Loss(strong_threshold=0.97).cuda(),
                 "contrast_loss": mix_label.Contrast_Loss(strong_threshold=0.8, num_queries=64, num_negatives=128, temp=0.5, alpha=0.99).cuda()}
    mix_label.prototypes = torch.zeros(C, 256).cuda()          # `global prototypes` of main() (mix_label.py:91-93), read by train()
    optimizer = torch.optim.SGD(model.module.model.parameters(), lr=1e-3, weight_decay=5e-4, momentum=0.9, nesterov=True)
    g = torch.Generator().manual_seed(5)
    mean = torch.tensor([0.485, 0.456, 0.406]).view(1, 3, 1, 1)
    std = torch.tensor([0.229, 0.224, 0.225]).view(1, 3, 1, 1)
    images = (torch.rand(2 * B * iters, 3, H, W, generator=g) - mean) / std
    labels = torch.randint(0, C, (2 * B * iters, 1, H // 16 + 1, W // 16 + 1), generator=g).float()
    labels = F.interpolate(labels, size=(H, W), mode="nearest")[:, 0].long()
    ds_l = TensorDataset(images[:B * iters], labels[:B * iters])
    ds_u = TensorDataset(images[B * iters:], labels[B * iters:])
    l_loader = DataLoader(ds_l, batch_size=B, sampler=DistributedSampler(ds_l, num_replicas=1, rank=0), drop_last=True)
    u_loader = DataLoader(ds_u, batch_size=B, sampler=DistributedSampler(ds_u, num_replicas=1, rank=0), drop_last=True)
    scheduler = PolyLR(optimizer, 100, min_lr=1e-4)
    sche_d = RampdownScheduler(begin_epoch=0, max_epoch=200, current_epoch=0, max_value=1.0, min_value=0, ramp_mult=-5.0)
    w_before = [p.detach().clone() for p in list(model.module.model.parameters())[-4:]]
    mix_label.train(l_loader, u_loader, model, optimizer, criterion, 0, scheduler, sche_d, config, args)
    last = criterion["contrast_loss"].last
    assert last is not None and last["rows_from_cache"] is True and last["rows_cache_mode"] == "verify"
    assert int(last["ws"].meta[css_b200._lib.META_ROWS_STALE].item()) == 0
    assert model.module.step == iters
    assert torch.isfinite(mix_label.prototypes).all().item() and mix_label.prototypes.abs().sum().item() > 0
    assert any(not torch.equal(a, b) for a, b in zip(w_before, list(model.module.model.parameters())[-4:]))
