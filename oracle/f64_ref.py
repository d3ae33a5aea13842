"""Float64 restatements of the CUDA kernels' operations, run with torch on whatever device the inputs live on.

TEST INFRASTRUCTURE, like css_oracle.py: only tests/ import it.  css_oracle.py rounds in fp32 the way the kernels do, so a
comparison against it shows whether the kernels follow the reference's arithmetic; these float64 versions measure the real
error of the fp32 results instead.  Gradients come from float64 autograd on the restated forward, never from the
closed-form formula the kernels use.  Selection lists and draws are integer work that other tests check exactly: the
callers take them from Contrast_Loss.selection() / sample_indices().  Reference lines are relative to the reference root
(WangChangqi98/CSS).
"""
import torch
import torch.nn.functional as F

f64 = torch.float64


def cos_sim_map(rep, prototypes):
    """Cosine map, ddp_model.py:104-110: F.normalize (x / max(||x||, 1e-12)) of every pixel and prototype row, then mm.
    rep [B,D,h,w], prototypes [C,D] -> [B,C,h,w] float64.  A zero prototype row gives 0."""
    x = F.normalize(rep.to(f64).permute(0, 2, 3, 1), dim=-1)             # :105-106
    p = F.normalize(prototypes.to(f64), dim=-1)                          # :107
    return (x @ p.T).permute(0, 3, 1, 2).contiguous()                    # :108-110


def proto_softmax_sim(rep, prototypes, temp):
    """Student softmax-similarity map, ddp_model.py:147-154: softmax(cos / temp) over the classes."""
    return torch.softmax(cos_sim_map(rep, prototypes) / temp, dim=1)


def upsample_softmax_max(x, out_hw, temp=None):
    """ddp_model.py:111-114: F.interpolate(bilinear, align_corners=True) to the crop size, softmax (of x / temp when a
    temperature is given), max over the classes.  Returns (conf, label, top-2 margin of the softmax), all [B,H,W]."""
    up = F.interpolate(x.to(f64), size=tuple(out_hw), mode="bilinear", align_corners=True)    # :111 / :113
    if temp is not None:
        up = up / temp                                                                        # :112
    p = torch.softmax(up, dim=1)
    conf, label = p.max(dim=1)                                                                # :112 / :114
    if p.shape[1] == 1:
        margin = torch.full_like(conf, float("inf"))
    else:
        top2 = p.topk(2, dim=1).values
        margin = top2[:, 0] - top2[:, 1]
    return conf, label, margin


def _cosine_rows(a, b, eps=1e-8):
    """torch.cosine_similarity (>= 1.12) along the last dim: each norm clamped at eps separately."""
    na = torch.linalg.vector_norm(a, dim=-1, keepdim=True).clamp_min(eps)
    nb = torch.linalg.vector_norm(b, dim=-1, keepdim=True).clamp_min(eps)
    return ((a / na) * (b / nb)).sum(-1)


def contrast_loss(rep, label, mask, prototypes, sel, anchor_idx, neg_idx, *, temp, alpha):
    """Contrast_Loss.forward (loss.py:75-149) in float64 with the draws fixed, and d loss / d rep by float64 autograd.

    rep [B2,D,h,w]; label [B2,C,h,w]; mask [B2,1,h,w]; prototypes [C,D] (read, not modified); sel: Contrast_Loss.selection()
    (present classes, valid / hard pixel ids per slot); anchor_idx [C,Q] and neg_idx [C,Q,Nn]: the slot-major draws
    (index into the slot's hard list / into the rotated concatenation of the other slots' valid lists).
    Returns (loss, grad_rep, updated prototypes [C,D]), float64.  As in the reference, only the anchors carry gradient: the
    prototype update, the positives and the negatives are computed without it (loss.py:100-109,131-144)."""
    B2, D, h, w = rep.shape
    dev = rep.device
    r = rep.detach().to(f64).requires_grad_(True)
    x = r.permute(0, 2, 3, 1).reshape(-1, D)                                           # :85
    xd = x.detach()
    valid_all = (label.to(f64) * mask.to(f64)).permute(0, 2, 3, 1).reshape(-1, label.shape[1])   # :80
    protos = prototypes.detach().to(f64).clone()
    present = sel["present"]
    V = len(present)
    proto_rep = []
    for c in present:                                                                  # :93-109
        mean = xd[valid_all[:, c] != 0].mean(0)                                        # :102
        if float(prototypes[c].sum()) == 0:                                            # :103 (tested on the fp32 buffer)
            protos[c] = mean                                                           # :105
        else:
            protos[c] = alpha * protos[c] + (1 - alpha) * mean                         # :108
        proto_rep.append(protos[c])
    if V <= 1:                                                                         # :116-117
        return torch.zeros((), dtype=f64, device=dev), torch.zeros_like(r), protos
    ids = [torch.as_tensor(v, dtype=torch.long, device=dev) for v in sel["valid_ids"]]
    loss = torch.zeros((), dtype=f64, device=dev)
    for k in range(V):                                                                 # :124
        if sel["n_hard"][k] == 0:                                                      # :125,129-130
            continue
        hard = torch.as_tensor(sel["hard_ids"][k], dtype=torch.long, device=dev)
        a = x[hard[anchor_idx[k].long()]]                                              # :127-128  [Q,D]
        negcat = torch.cat(ids[k + 1:] + ids[:k])                                      # :141
        neg = xd[negcat[neg_idx[k].long()]]                                            # :142       [Q,Nn,D]
        cand = torch.cat([proto_rep[k].expand(a.shape[0], 1, D), neg], dim=1)          # :143-144  [Q,1+Nn,D]
        z = _cosine_rows(a[:, None, :], cand) / temp                                   # :146
        loss = loss + F.cross_entropy(z, torch.zeros(a.shape[0], dtype=torch.long, device=dev))   # :147
    loss = loss / V                                                                    # :149
    (grad,) = torch.autograd.grad(loss, r)
    return loss.detach(), grad, protos


def attention_threshold_loss(pred, pseudo_label, logits, strong_threshold):
    """Attention_Threshold_Loss.forward (loss.py:48-64) in float64, and d loss / d pred by float64 autograd.
    pred [B,C,H,W]; pseudo_label [B,H,W] int (-1 = ignored); logits [B,H,W] confidences.  Returns (loss, grad_pred)."""
    B = pred.shape[0]
    p = pred.detach().to(f64).requires_grad_(True)
    lab = pseudo_label.long()
    weighting = ((logits.reshape(B, -1) >= strong_threshold).sum(-1).to(f64)
                 / (lab.reshape(B, -1) >= 0).sum(-1).to(f64))                            # :55-56
    ce = F.cross_entropy(p, lab, ignore_index=-1, reduction="none")                       # :58-59
    keep = ce.detach() > 0                                                                # :60
    # the weighting multiplies the selected pixels only: an image without valid pixels has weighting 0/0 and no selected pixel
    wmap = weighting[:, None, None].expand_as(ce)
    out = (wmap[keep] * ce[keep]).mean()                                                  # :61-64
    (grad,) = torch.autograd.grad(out, p)
    return out.detach(), grad
