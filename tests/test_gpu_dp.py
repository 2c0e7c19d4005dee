"""Data-parallel HeadStep on 2 GPUs (NCCL) against the single-GPU step on the concatenated batch
(SURVEY 8d config 4 / 8e): the all-reduced int64 confusion matrix and valid count are bit-identical, the mean
loss and the summed prototype gradient agree to fp32 round-off.  Skipped with fewer than 2 GPUs."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, out):
    import torch.distributed as dist
    from lc2is_b200 import synthetic
    from lc2is_b200.step import HeadStep
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    dev = torch.device("cuda", rank)
    Bg, h, H, C = 8, 32, 512, 150
    v = synthetic.make_patch_embeddings(Bg, h * h, 512)
    t = synthetic.make_prototypes(C, 512)
    labels = synthetic.make_labels(Bg, H, H, C, ignore_frac=0.1)
    labels[Bg // 2:, :200] = 0                               # unequal valid counts per rank
    b = Bg // world
    step = HeadStep(b, h, h, H, H, C, ignore_index=0, device=dev, distributed=True)
    vd, td, ld = v[rank * b:(rank + 1) * b].to(dev), t.to(dev), labels[rank * b:(rank + 1) * b].to(dev)
    for _ in range(2):                                       # the confusion matrix accumulates over calls
        step(vd, td, ld)                                     # (the bucket all-reduce of call 1 runs behind call 2)
    step.flush()                                             # ... and the last call's here
    cm_global = step.global_confmat().clone()                # ONE int64 all-reduce for both steps
    torch.cuda.synchronize()
    if rank == 0:
        ref = HeadStep(Bg, h, h, H, H, C, ignore_index=0, device=dev, distributed=False)
        ref(v.to(dev), t.to(dev), labels.to(dev))
        torch.cuda.synchronize()
        res = {
            "cm_equal": bool(torch.equal(cm_global, 2 * ref.confmat)),
            "nv": (int(step.n_valid), int(ref.n_valid)),
            "loss": (float(step.loss), float(ref.loss)),
            "gt_err": float((step.grad_t - ref.grad_t).abs().max() / ref.grad_t.abs().max()),
            "gv_err": float((step.grad_v.float() - ref.grad_v[:b].float()).abs().max() / ref.grad_v.float().abs().max()),
        }
        torch.save(res, out)
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_step_matches_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    out = str(tmp_path / "res.pt")
    mp.spawn(_worker, args=(2, 29533, out), nprocs=2, join=True)
    r = torch.load(out)
    assert r["cm_equal"], "all-reduced confusion matrix differs from the single-GPU matrix"
    assert r["nv"][0] == r["nv"][1]
    assert abs(r["loss"][0] - r["loss"][1]) <= 2e-6 * abs(r["loss"][1])
    assert r["gt_err"] < 2e-3, r                             # bf16 GEMM operands, different split-K partition
    assert r["gv_err"] < 2e-2, r
