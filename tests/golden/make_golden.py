"""Generate the committed golden fixtures by running the REFERENCE itself.

Needs a checkout of the reference project (LC2IS), read-only:

    python tests/golden/make_golden.py /path/to/LC2IS

It imports the reference modules that import cleanly (``model.loss``,
``model.text_patch`` - SURVEY 8c) and restates, verbatim with live torch ops, the head
lines of ``model/final.py:37-44`` (final.py itself cannot be imported: it needs the
un-vendored ``model.DenseCLIP`` checkout).  ``metrics.py`` cannot be imported either
(torchmetrics is missing), so the confusion-matrix fixtures are produced by a naive
pure-Python double loop written here, independent of ``oracle/``.

The fixtures are committed, so the tests need no reference checkout.  Every fixture stays under 1 MB:
head_final.pt keeps the upsampled map of every 4th class only.
"""
import os
import sys

import torch
import torch.nn.functional as F
from einops import rearrange

OUT = os.path.dirname(os.path.abspath(__file__))


def main(ref):
    sys.path.insert(0, ref)
    from model.loss import AuxiliaryLoss            # reference class, loss.py:12-21
    from model.text_patch import TextToPatch        # reference class, text_patch.py:4-18

    protos = torch.load(os.path.join(ref, "model", "ade20k_prototypes.pt")).detach().float()
    g = torch.Generator().manual_seed(1024)

    # ---- 1. head lines of final.py:37-44 (x4 main head) and :262-268 (aux head) ----------
    B, h, D = 2, 8, 512
    v = torch.randn(B, h * h, D, generator=g)
    t = protos.expand(B, -1, -1)                                        # final.py:31
    vm = rearrange(v, "b (h w) c -> b c h w", h=h)                      # final.py:37
    vn = F.normalize(vm, dim=1, p=2)                                    # final.py:41
    tn = F.normalize(t, dim=2, p=2)                                     # final.py:42
    score_low = torch.einsum('bchw,bkc->bkhw', vn, tn)                  # final.py:43
    score_up = F.interpolate(input=score_low, mode="bilinear", scale_factor=4)  # final.py:44
    raw = torch.matmul(v, protos.transpose(1, 0))                       # model.py:50
    raw = rearrange(raw, "b (h w) c -> b c h w", h=h)                   # model.py:53
    up_classes = torch.arange(0, score_up.shape[1], 4)
    torch.save(dict(v=v, score_low=score_low, score_up=score_up[:, up_classes].clone(), raw=raw,
                    up_classes=up_classes),                             # t = bundled prototypes
               os.path.join(OUT, "head_final.pt"))

    # ---- 2. AuxiliaryLoss (reference class) fwd + autograd bwd ------------------------------
    cases = {}
    for name, (b, c, hh, H, ign) in {
        "x4_c151_ign0": (2, 151, 8, 32, 0),
        "x16_c151_ign0": (2, 151, 2, 32, 0),
        "x4_c150_noign": (1, 150, 8, 32, -100),
        "x2_c7_ign3": (2, 7, 5, 10, 3),        # non-multiple-of-4 scale -> generic path
        "x3p2_c5_ign0": (1, 5, 5, 16, 0),      # non-integer scale 3.2
    }.items():
        low = torch.randn(b, c, hh, hh, generator=g).requires_grad_(True)
        lab = torch.randint(0, c, (b, H, H), generator=g)
        crit = AuxiliaryLoss(ignore_index=ign)
        loss = crit(low, lab)
        loss.backward()
        cases[name] = dict(low=low.detach().clone(), labels=lab, ignore_index=ign,
                           loss=loss.detach().clone(), grad=low.grad.detach().clone())
    # all pixels ignored -> nan loss (0/0), zero... record what the reference does
    low = torch.randn(1, 4, 4, 4, generator=g).requires_grad_(True)
    lab = torch.zeros(1, 16, 16, dtype=torch.int64)
    loss = AuxiliaryLoss(ignore_index=0)(low, lab)
    loss.backward()
    cases["all_ignored"] = dict(low=low.detach().clone(), labels=lab, ignore_index=0,
                                loss=loss.detach().clone(), grad=low.grad.detach().clone())
    torch.save(cases, os.path.join(OUT, "aux_loss.pt"))

    # ---- 3. TextToPatch (reference class) ----------------------------------------------------
    torch.manual_seed(1024)
    m = TextToPatch(img_in=48, text_in=32, out=64)
    img = torch.randn(2, 9, 48, generator=g)
    txt = torch.randn(11, 32, generator=g)
    tf, vf = m(img, txt)
    torch.save(dict(state=m.state_dict(), img=img, text=txt, t_feature=tf.detach(), v_feature=vf.detach()),
               os.path.join(OUT, "text_patch.pt"))

    # ---- 4. confusion matrix / per-image IoU by naive loops (independent of oracle/) ---------
    C, hh = 6, 6
    out = torch.randint(-512, 513, (3, C, hh, hh), generator=g).float() / 64.0
    lab = torch.randint(0, C, (3, hh, hh), generator=g)
    up = F.interpolate(out, mode="bicubic", scale_factor=4)               # metrics.py:89
    labu = F.interpolate(lab.view(-1, 1, hh, hh).float(), mode="nearest", scale_factor=4).squeeze(1).long()  # :90
    pred = torch.softmax(up, dim=1).argmax(dim=1)                         # Softmax2d + argmax
    cms = torch.zeros(3, C, C, dtype=torch.int64)
    for n in range(3):
        for y in range(4 * hh):
            for x in range(4 * hh):
                cms[n, int(labu[n, y, x]), int(pred[n, y, x])] += 1
    per_img = []
    for n in range(3):
        ious = []
        for k in sorted(set(labu[n].flatten().tolist())):
            if k == 0:
                continue
            inter = int(cms[n, k, k]); union = int(cms[n, k].sum() + cms[n, :, k].sum() - inter)
            ious.append(inter / union if union else 0.0)
        per_img.append(sum(ious) / len(ious))
    glob = cms.sum(0).clone(); glob[0] = 0
    gi = []
    for k in range(1, C):
        inter = int(glob[k, k]); union = int(glob[k].sum() + glob[:, k].sum() - inter)
        gi.append(inter / union if union else 0.0)
    torch.save(dict(outputs=out, labels=lab, pred=pred, confmats=cms,
                    miou_label=float(sum(per_img) / len(per_img)), miou_global=float(sum(gi) / len(gi))),
               os.path.join(OUT, "metrics_small.pt"))
    # ---- 5. ContrastiveLoss (reference class, loss.py:39-64) fwd + autograd bwd of the total ----------------
    from model.loss import ContrastiveLoss
    g5 = torch.Generator().manual_seed(1029)
    cases = {}
    for name, (b, hh, ign, hi) in {
        "h8": (2, 8, -100, 151),                      # ignore_index >= 0 raises in the reference (float target)
        "h6_ign_m1": (1, 6, -1, 151),
        "h16_few_classes": (2, 16, -100, 5),          # long label runs: several rows of a column share a class
    }.items():
        out = (torch.randn(b, hh * hh, 151, generator=g5) * 3).requires_grad_(True)
        lab = torch.randint(0, hi, (b, hh, hh), generator=g5)
        total, lv, lt = ContrastiveLoss(ignore_index=ign)(out, lab)
        total.backward()
        cases[name] = dict(outputs=out.detach().clone(), labels=lab, ignore_index=ign, total=total.detach().clone(),
                           loss_visual=lv.detach().clone(), loss_textual=lt.detach().clone(),
                           grad=out.grad.detach().clone())
    torch.save(cases, os.path.join(OUT, "contrastive.pt"))

    print("golden fixtures written to", OUT)
    for f in sorted(os.listdir(OUT)):
        if f.endswith(".pt"):
            print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/make_golden.py /path/to/LC2IS")
    main(sys.argv[1])
