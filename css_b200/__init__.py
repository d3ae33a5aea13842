"""css_b200 -- B200-native (sm_100a) representation-space hot path of CSS ("Space Engage", ICCV'23).

Public surface (mirrors the reference's names for this path):
    Contrast_Loss                                   generalframeworks/loss/loss.py:66-149
    Attention_Threshold_Loss                        generalframeworks/loss/loss.py:48-64   (SURVEY.md 8(f)-3)
    ProbOhemCrossEntropy2d                          generalframeworks/loss/loss.py:8-46    (DESIGN.md f-5, supervised OHEM CE)
    Model_ori_pseudo, Model_mix, Model_cross        generalframeworks/networks/ddp_model.py:8-239
    ops.cos_sim_map / proto_softmax_sim / pseudo_labels / rep_pseudo_label / cls_pseudo_label / mix_fuse / threshold_glue
    aug.batch_transform{,_2,_3}, aug.generate_cut_gather{,_2,_3}     dataset_helpers/VOC.py:312-477 for the label / confidence maps
                                                    (SURVEY.md 8(f)-2; imported on demand: needs torchvision + Pillow)
    comm.PeerStatsReducer                           the class-statistics exchange over NVLink peer memory (one node)
    install.install()                               monkey-patches an unmodified reference checkout
Importing the package does not load the CUDA library; the first op call does, and raises if it is missing.
"""
from .loss import Contrast_Loss, Attention_Threshold_Loss, ProbOhemCrossEntropy2d, allreduce_class_stats   # noqa: F401
from .models import Model_ori_pseudo, Model_mix, Model_cross     # noqa: F401
from . import ops                                                # noqa: F401

__version__ = "0.1.0"
