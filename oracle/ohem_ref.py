"""Test-only restatement of the reference's ProbOhemCrossEntropy2d (generalframeworks/loss/loss.py:8-46), pure torch.

The forward is the reference's, statement by statement (it synchronises with the host three times and cannot be captured in
a CUDA graph).  The one addition is `self.last`: the threshold used and the final kept mask, recorded without changing any
computation, so that tests can compare the selection of css_b200.ProbOhemCrossEntropy2d exactly.
tests/test_ohem_host.py checks this module against the reference's own class when a checkout of it is available.
"""
import logging

import torch
import torch.nn as nn
import torch.nn.functional as F

logger = logging.getLogger(__name__)

CLASS_WEIGHTS = [0.8373, 0.918, 0.866, 1.0345, 1.0166, 0.9969, 0.9754, 1.0489, 0.8786, 1.0023,
                 0.9539, 0.9843, 1.1116, 0.9037, 1.0865, 1.0955, 1.0865, 1.1529, 1.0507]


class ProbOhemCrossEntropy2d(nn.Module):
    def __init__(self, ignore_index, reduction='mean', thresh=0.6, min_kept=256, down_ratio=1, use_weight=False):
        super(ProbOhemCrossEntropy2d, self).__init__()
        self.ignore_index = ignore_index
        self.thresh = float(thresh)
        self.min_kept = int(min_kept)
        self.down_ratio = down_ratio
        if use_weight:
            weight = torch.FloatTensor(CLASS_WEIGHTS)
            self.criterion = nn.CrossEntropyLoss(reduction=reduction, weight=weight, ignore_index=ignore_index)
        else:
            self.criterion = nn.CrossEntropyLoss(reduction=reduction, ignore_index=ignore_index)
        self.last = None

    def forward(self, pred, target):
        b, c, h, w = pred.size()
        target = target.view(-1)
        valid_mask = target.ne(self.ignore_index)
        target = target * valid_mask.long()
        num_valid = valid_mask.sum()
        prob = F.softmax(pred, dim=1)
        prob = (prob.transpose(0, 1)).reshape(c, -1)
        threshold = None                                       # diagnostics only: None = no OHEM selection ran
        if self.min_kept > num_valid:
            logger.info('Labels: {}'.format(num_valid))
        elif num_valid > 0:
            prob = prob.masked_fill_(~valid_mask, 1)
            mask_prob = prob[target, torch.arange(len(target), dtype=torch.long)]
            threshold = self.thresh
            if self.min_kept > 0:
                index = mask_prob.argsort()
                threshold_index = index[min(len(index), self.min_kept) - 1]
                if mask_prob[threshold_index] > self.thresh:
                    threshold = mask_prob[threshold_index]
                kept_mask = mask_prob.le(threshold)
                target = target * kept_mask.long()
                valid_mask = valid_mask * kept_mask
            else:
                threshold = None
        target = target.masked_fill_(~valid_mask, self.ignore_index)
        target = target.view(b, h, w)
        self.last = dict(valid_mask=valid_mask.view(b, h, w).clone(), num_valid=num_valid, threshold=threshold)
        return self.criterion(pred, target)
