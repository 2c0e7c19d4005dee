"""Time the weighted / label-smoothed form of the fused upsample + cross-entropy (lc2is_upsample_ce_fwd_bwd_ex with class
weights and eps = 0.1) against the unweighted call (lc2is_upsample_ce_fwd_bwd), alternating the two in one process with
CUDA events: ROUNDS rounds of ITERS launches of each, after a warm-up, per shape.  The torch route a user would take
otherwise (F.interpolate + F.cross_entropy(weight, label_smoothing) + backward, on the GPU) is timed for context, on as
many images as keep the upsampled map under 4 GB, scaled to the batch.  Inputs are not rotated: the low-resolution logits
(10 - 217 MB) and labels are the working set, read from L2 where they fit, for both variants alike.
Prints the card's name and power limit and one JSON line per shape; --out FILE also writes all of it as one JSON file
(results: profiles/r04_ce_weighted.md, raw: profiles/r04_ce_weighted_times.json).

    python tools/time_ce_weighted.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

from lc2is_b200 import ops, synthetic

DEV = "cuda"
ROUNDS, ITERS, TORCH_ITERS = 5, 50, 10
# name, B, C, h, H, which kernel the geometry selects
SHAPES = [
    ("x16 G-A", 16, 150, 32, 512, "k2_strip_kernel<16>"),
    ("x8", 16, 150, 64, 512, "k2_strip_kernel<8>"),
    ("x4 G-B", 16, 150, 128, 512, "k2_fast_kernel"),
    ("x16 C=847", 8, 847, 64, 1024, "k2_strip_gtaps_kernel<16>"),
    ("generic 24->120", 4, 150, 24, 120, "k2_generic_kernel"),          # scale 5: not a power of two
]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def time_launches(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / n               # us per launch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the card and all results to this JSON file")
    args = ap.parse_args()
    info = card()
    print("card (name, power limit, max SM clock):", info, flush=True)
    res = []
    for name, B, C, h, H, kernel in SHAPES:
        g = torch.Generator().manual_seed(71)
        low = (torch.randn(B, C, h, h, generator=g) * 2.0).to(DEV)
        labels = synthetic.make_labels(B, H, H, C, ignore_frac=0.1).to(DEV)
        w = (0.2 + 2.8 * torch.rand(C, generator=g)).to(DEV)
        gs = torch.tensor([1e-6], device=DEV)
        ls = torch.zeros(1, dtype=torch.float64, device=DEV)
        plain = lambda: ops.upsample_ce(low, labels, 0, gs, loss_sum=ls)
        weighted = lambda: ops.upsample_ce(low, labels, 0, gs, loss_sum=ls, weight=w, label_smoothing=0.1)
        for fn in (plain, weighted):
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        tp, tw = [], []
        for _ in range(ROUNDS):
            tp.append(time_launches(plain, ITERS))
            tw.append(time_launches(weighted, ITERS))

        # torch route on the first nb images (the upsampled map and its gradient are 4 x B*C*H*H bytes each), scaled to B
        nb = max(1, min(B, int(4e9 // (C * H * H * 4))))
        x = low[:nb].clone().requires_grad_(True)

        def torch_route():
            x.grad = None
            up = F.interpolate(x, size=(H, H), mode="bilinear", align_corners=False)
            F.cross_entropy(up, labels[:nb], weight=w, ignore_index=0, label_smoothing=0.1).backward()
        torch_route()
        torch.cuda.synchronize()
        tt = time_launches(torch_route, TORCH_ITERS) * B / nb
        x = None
        torch.cuda.empty_cache()
        med = lambda v: sorted(v)[len(v) // 2]
        r = dict(shape=name, B=B, C=C, h=h, H=H, kernel=kernel, launches=ROUNDS * ITERS,
                 unweighted_us=round(med(tp), 1), weighted_us=round(med(tw), 1),
                 ratio=round(med(tw) / med(tp), 3),
                 unweighted_rounds_us=[round(v, 1) for v in tp], weighted_rounds_us=[round(v, 1) for v in tw],
                 torch_route_us=round(tt, 1), torch_route_images=nb)
        res.append(r)
        print(json.dumps(r), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(dict(card=info, results=res), f, indent=1)


if __name__ == "__main__":
    main()
