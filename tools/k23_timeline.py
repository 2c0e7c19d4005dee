"""Per-warp timeline of k23_rc_kernel from an instrumented build (csrc built with -DRC_STAMPS; development aid).
build:  nvcc ... -DRC_STAMPS -c k23_rowclass.cu && relink;  usage: python tools/k23_timeline.py [B]
Per warp RC_STAMP_SLOTS = 32 stamps: [0] start, then (class phase starts, job ends) per job, [31] = stamps taken."""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from lc2is_b200 import synthetic, _lib
from lc2is_b200.step import HeadStep
SLOTS = 32
B = int(sys.argv[1]) if len(sys.argv) > 1 else 16
h, H, C, D = 32, 512, 150, 512
V = synthetic.make_patch_embeddings(B, h * h, D).cuda(); L = synthetic.make_labels(B, H, H, C, ignore_frac=0.1).cuda()
t = synthetic.make_prototypes(C, D).cuda()
hs = HeadStep(B, h, h, H, H, C, ignore_index=0)
for _ in range(5): hs(V, t, L)
torch.cuda.synchronize()
buf = np.zeros(148 * 16 * SLOTS, dtype=np.uint64)
rc = _lib.lib.lc2is_debug_stamps(buf.ctypes.data_as(ctypes.c_void_p)); assert rc == 0, rc
S = buf.reshape(148 * 16, SLOTS).astype(np.int64)
n = S[:, SLOTS - 1]; ok = n >= 3
t0 = S[ok, 0].min()
start = S[ok, 0] - t0
ends = np.array([S[i, n[i] - 1] - t0 for i in np.nonzero(ok)[0]])
print(f"warps {ok.sum()}  start spread {start.max()/1e3:.1f} us  kernel span {ends.max()/1e3:.1f} us")
print("last-stamp (warp end) percentiles us:", [round(float(np.percentile(ends, p)) / 1e3, 1) for p in (0, 5, 25, 50, 75, 95, 100)])
jobs = (n - 1) // 2
print("jobs per warp histogram:", {int(k): int((jobs[ok] == k).sum()) for k in np.unique(jobs[ok])})
# per job ordinal: duration (end - previous end), row-phase share
for j in range(int(jobs[ok].max())):
    sel = ok & (jobs > j)
    prev = S[sel, 0] if j == 0 else S[sel, 2 * j]
    mid, end = S[sel, 2 * j + 1], S[sel, 2 * j + 2]
    d = (end - prev) / 1e3; r = (mid - prev) / 1e3
    print(f"job #{j}: n={sel.sum():5d}  duration mean {d.mean():6.1f} us (p5 {np.percentile(d,5):.1f}, p95 {np.percentile(d,95):.1f})  up-to-class-phase {r.mean():6.1f} us  class phase {(d-r).mean():6.1f} us  starts at {((prev - t0)/1e3).mean():6.1f} us")
# busy warps over time
grid = np.arange(0, ends.max(), 5000)
busy = [(ends > g).sum() for g in grid]
print("busy warps every 5 us:", list(zip((grid / 1e3).astype(int).tolist(), busy))[-20:])
