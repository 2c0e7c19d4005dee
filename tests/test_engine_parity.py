"""Engine (lc2is_b200/engine.py) under data parallelism and CUDA graphs against the single-process run.

The reference of every test is the same model trained by one process on the concatenated batches (the ranks' j-th
batches together are batch j), with plain torch.  On the CPU (gloo, float64, SGD) the ranks see shards of unequal size
and very unequal ignored fractions, criteria with class weights or reduction='sum', differently seeded replicas,
evaluation shards of which one is empty, and train loaders of different lengths.  On the GPU the head-shaped model
(projection -> cosine_logits (K1/K1b) -> AuxiliaryLoss (K2)) runs graphed with short batches, against the eager Engine
and a float64 CPU autograd run, and on two devices (NCCL) against one.

Multi-process tests run in spawned processes; a rank that fails reports its traceback at once, a rank that hangs fails
the test at the timeout, and no child outlives the test."""
import os
import queue
import socket
import time
import traceback

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F
from torch import nn

from lc2is_b200 import dp
from lc2is_b200.engine import Engine


# ---- harness -------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _entry(fn, rank, world, port, backend, q, args):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.set_num_threads(1)
    try:
        dp.init_distributed(backend)
        q.put((rank, "ok", fn(rank, world, *args)))
    except BaseException:  # noqa: BLE001  (reported to the parent, which fails the test)
        q.put((rank, "error", traceback.format_exc()))
    finally:
        if dist.is_initialized():
            dist.destroy_process_group()


def _spawn(fn, world, *args, backend="gloo", timeout=120.0):
    """Run fn(rank, world, *args) on `world` ranks; -> {rank: result}.  Fails on the first rank that raises and on a
    timeout; every child is gone when it returns."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_entry, args=(fn, r, world, port, backend, q, args)) for r in range(world)]
    try:
        for p in ps:
            p.start()
        got, deadline = {}, time.monotonic() + timeout
        while len(got) < world:
            try:
                rank, status, payload = q.get(timeout=max(0.1, deadline - time.monotonic()))
            except queue.Empty:
                pytest.fail(f"ranks {sorted(set(range(world)) - set(got))} did not finish within {timeout} s (hang)")
            if status != "ok":
                pytest.fail(f"rank {rank} raised:\n{payload}")
            got[rank] = payload
        for p in ps:
            p.join(timeout=30)
        return got
    finally:
        for p in ps:
            if p.is_alive():
                p.terminate()
        for p in ps:
            p.join(timeout=10)
            if p.is_alive():
                p.kill()
                p.join()


def _rel(a, b):
    a, b = torch.as_tensor(a, dtype=torch.float64), torch.as_tensor(b, dtype=torch.float64)
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def _state_np(model):
    return {k: v.detach().cpu().numpy().copy() for k, v in model.state_dict().items()}


class _LoggedEngine(Engine):
    """Keeps what every log() returns (log_step=1: the per-step losses)."""

    def log(self):
        m = super().log()
        self.history = getattr(self, "history", []) + [m]
        return m


# ---- CPU: float64 two-head model, gloo ------------------------------------------------------------------------------
C, H = 5, 8
_WEIGHT = torch.linspace(0.5, 2.0, C, dtype=torch.float64)
_LR = dict(mean=0.1, weight=0.1, sum=1e-3)


class TwoHead(nn.Module):
    """{'image': [B,3,H,W]} -> {'outputs', 'low_score_map'}: the main and the aux criterion each see their own map."""

    def __init__(self):
        super().__init__()
        self.conv = nn.Conv2d(3, C, 1)
        self.aux = nn.Conv2d(3, C, 3, padding=1)

    def forward(self, inputs):
        x = inputs["image"]
        return dict(outputs=self.conv(x), low_score_map=self.aux(x))


def _model(seed):
    torch.manual_seed(seed)
    return TwoHead().double()


def _criteria(case):
    """Main: ignore_index=0 (mean, class-weighted or summed); aux: ignore_index=-100, mean (x0.4 in Engine)."""
    main = dict(mean=lambda: nn.CrossEntropyLoss(ignore_index=0),
                weight=lambda: nn.CrossEntropyLoss(weight=_WEIGHT, ignore_index=0),
                sum=lambda: nn.CrossEntropyLoss(ignore_index=0, reduction="sum"))[case]()
    return main, nn.CrossEntropyLoss()


def _global_batches(n_steps, n_img, world, seed, ignore_frac0=0.9):
    """n_steps batches of n_img images; on rank 0's images a fraction ignore_frac0 of the labels is 0 (ignored by the
    main criterion), so the ranks' valid counts differ a lot."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n_steps):
        img = torch.randn(n_img, 3, H, H, generator=g, dtype=torch.float64)
        lab = torch.randint(1, C, (n_img, H, H), generator=g)
        a, b = dp.shard_range(n_img, 0, world)
        lab[a:b][torch.rand(b - a, H, H, generator=g) < ignore_frac0] = 0
        out.append((img, lab))
    return out


def _shard(batches, rank, world):
    res = []
    for img, lab in batches:
        a, b = dp.shard_range(img.shape[0], rank, world)
        if b > a:
            res.append((dict(image=img[a:b], label=lab[a:b]), None))
    return res


def _reference(case, batches, seed):
    """One process, plain torch: -> (state, mean main loss, mean 0.4 * aux loss over the steps)."""
    m = _model(seed)
    crit, aux = _criteria(case)
    opt = torch.optim.SGD(m.parameters(), lr=_LR[case])
    mains, auxs = [], []
    for img, lab in batches:
        opt.zero_grad()
        o = m(dict(image=img))
        lm, la = crit(o["outputs"], lab), aux(o["low_score_map"], lab) * 0.4
        (lm + la).backward()
        opt.step()
        mains.append(float(lm.detach())); auxs.append(float(la.detach()))
    return _state_np(m), float(np.mean(mains)), float(np.mean(auxs))


def _train_worker(rank, world, case, n_img, n_steps, seed_per_rank):
    m = _model(rank if seed_per_rank else 0)
    crit, aux = _criteria(case)
    loader = _shard(_global_batches(n_steps, n_img, world, 5), rank, world)
    eng = Engine("p", m, torch.optim.SGD(m.parameters(), lr=_LR[case]), crit, aux_criterion=aux, device="cpu",
                 train_loader=loader, logger=None, save_step=10 ** 9, log_step=n_steps)
    metrics, _ = eng.train()
    return dict(state=_state_np(m), train_loss=metrics["train_loss"], train_aux_loss=metrics["train_aux_loss"])


@pytest.mark.parametrize("world,n_img,case", [(2, 5, "mean"), (3, 7, "mean"), (2, 5, "sum"), (3, 7, "weight")])
def test_dp_train_matches_single_process(world, n_img, case):
    """Unequal shards (5 images over 2 ranks, 7 over 3), 90 % of rank 0's labels ignored by the main criterion, an aux
    criterion with another ignore_index: every rank's weights and the logged losses are the single-process ones."""
    n_steps = 3
    got = _spawn(_train_worker, world, case, n_img, n_steps, False)
    ref_state, ref_main, ref_aux = _reference(case, _global_batches(n_steps, n_img, world, 5), 0)
    for r in range(world):
        for k, v in ref_state.items():
            assert _rel(got[r]["state"][k], v) <= 1e-10, (r, k, _rel(got[r]["state"][k], v))
        assert _rel(got[r]["train_loss"], ref_main) <= 1e-10, (r, got[r]["train_loss"], ref_main)
        assert _rel(got[r]["train_aux_loss"], ref_aux) <= 1e-10, (r, got[r]["train_aux_loss"], ref_aux)


def test_dp_ranks_seeded_differently_follow_rank0():
    """Replicas built from different seeds: the constructor's broadcast makes every rank train rank 0's weights."""
    world, n_img, n_steps = 2, 4, 3
    got = _spawn(_train_worker, world, "mean", n_img, n_steps, True)
    ref_state, ref_main, _ = _reference("mean", _global_batches(n_steps, n_img, world, 5), 0)
    for r in range(world):
        for k, v in ref_state.items():
            assert _rel(got[r]["state"][k], v) <= 1e-10, (r, k)
        assert _rel(got[r]["train_loss"], ref_main) <= 1e-10


def _eval_worker(rank, world):
    m = _model(0)
    crit, aux = _criteria("mean")
    img, lab = _global_batches(1, 2, world, 7)[0]          # 2 images over 3 ranks: rank 2's shard is empty
    seen = {}

    def compute_metrics(outputs, labels):
        seen.update(outputs=outputs.numpy().copy(), labels=labels.numpy().copy())
        return dict(n_images=int(outputs.shape[0]))
    eng = Engine("e", m, None, crit, aux_criterion=aux, device="cpu", eval_loader=_shard([(img, lab)], rank, world),
                 compute_metrics=compute_metrics, online_metrics=False, logger=None)
    return dict(metrics=eng.evaluate(), seen=seen)


def test_dp_eval_uneven_shards_with_an_empty_one():
    """Non-online evaluation, 2 images over 3 ranks: it finishes, compute_metrics gets the whole set, and eval_loss /
    eval_aux_loss are the losses of the one batch the single process sees."""
    world = 3
    got = _spawn(_eval_worker, world)
    img, lab = _global_batches(1, 2, world, 7)[0]
    m = _model(0)
    crit, aux = _criteria("mean")
    with torch.no_grad():
        o = m(dict(image=img))
        ref_loss, ref_aux = float(crit(o["outputs"], lab)), float(aux(o["low_score_map"], lab) * 0.4)
    for r in range(world):
        seen, met = got[r]["seen"], got[r]["metrics"]
        assert seen["outputs"].shape == (2, C, H, H), (r, seen["outputs"].shape)
        assert np.array_equal(seen["labels"], lab.numpy()), r
        assert _rel(seen["outputs"], o["outputs"]) <= 1e-12, r
        assert met["eval_n_images"] == 2
        assert _rel(met["eval_loss"], ref_loss) <= 1e-10, (r, met["eval_loss"], ref_loss)
        assert _rel(met["eval_aux_loss"], ref_aux) <= 1e-10, (r, met["eval_aux_loss"], ref_aux)


def _unequal_loader_worker(rank, world):
    m = _model(0)
    crit, aux = _criteria("mean")
    loader = _shard(_global_batches(3 - rank, 2 * world, world, 5), rank, world)   # 3 batches on rank 0, 2 on rank 1
    eng = Engine("u", m, torch.optim.SGD(m.parameters(), lr=0.1), crit, aux_criterion=aux, device="cpu",
                 train_loader=loader, logger=None, save_step=10 ** 9)
    try:
        eng.train()
    except RuntimeError as e:
        return str(e)
    return None


def test_dp_unequal_train_loader_lengths_raise_on_every_rank():
    got = _spawn(_unequal_loader_worker, 2, timeout=60.0)
    for r in range(2):
        assert got[r] is not None and "number of training steps" in got[r], (r, got[r])


def test_online_metrics_defaults_to_calling_compute_metrics():
    """A compute_metrics passed the way the reference's evaluate.py passes it is called."""
    m = _model(0)
    crit, aux = _criteria("mean")
    img, lab = _global_batches(1, 3, 1, 7)[0]
    calls = []

    def compute_metrics(outputs, labels):
        calls.append(tuple(outputs.shape))
        return dict(acc=float((outputs.argmax(1) == labels).double().mean()))
    eng = Engine("d", m, None, crit, aux_criterion=aux, device="cpu", eval_loader=[(dict(image=img, label=lab), None)],
                 compute_metrics=compute_metrics, logger=None)
    got = eng.evaluate()
    assert calls == [(3, C, H, H)] and "eval_acc" in got
    assert Engine("d", m, None, crit, device="cpu", logger=None).online_metrics      # no compute_metrics: online


# ---- GPU: head-shaped model (K1/K1b + K2) ----------------------------------------------------------------------------
HC, HD, HH = 12, 64, 8                                       # classes, embedding width, low-resolution grid


class HeadModel(nn.Module):
    """TextToPatch-like projection -> cosine logits; the low map is both 'outputs' and 'low_score_map'."""

    def __init__(self):
        super().__init__()
        self.visual = nn.Linear(32, HD)
        self.t = nn.Parameter(torch.randn(HC, HD))

    def forward(self, inputs):
        from lc2is_b200 import head
        low = head.cosine_logits(self.visual(inputs["patches"]), self.t, hw_shape=(HH, HH))
        return dict(outputs=low, low_score_map=low)


def _head_model(seed):
    torch.manual_seed(seed)
    return HeadModel()


def _head_batches(sizes, seed, ignore_frac=None):
    """Batches of the given sizes, labels on the x16 grid; ignore_frac[i]: fraction of image i's labels set to 0."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for b in sizes:
        lab = torch.randint(0, HC, (b, 16 * HH, 16 * HH), generator=g)
        if ignore_frac is not None:
            for i in range(b):
                lab[i][torch.rand(16 * HH, 16 * HH, generator=g) < ignore_frac[i]] = 0
        out.append((dict(patches=torch.randn(b, HH * HH, 32, generator=g), label=lab), None))
    return out


def _head_engine(model, loader, device, graph=False, max_epoch=1):
    from lc2is_b200.model.loss import AuxiliaryLoss
    crit = AuxiliaryLoss(ignore_index=0)
    return _LoggedEngine("h", model, torch.optim.SGD(model.parameters(), lr=0.5), crit, aux_criterion=crit,
                         device=device, train_loader=loader, logger=None, save_step=10 ** 9, log_step=1,
                         max_epoch=max_epoch, cuda_graph=graph)


def _head_reference(model, loader, max_epoch):
    """float64 CPU autograd of the same step: F.normalize + einsum, F.interpolate (bilinear) + F.cross_entropy."""
    p = {k: v.detach().double().clone().requires_grad_(True) for k, v in model.named_parameters()}
    losses = []
    for _ in range(max_epoch):
        for d, _m in loader:
            x, lab = d["patches"].double(), d["label"]
            v = F.normalize(x @ p["visual.weight"].T + p["visual.bias"], dim=-1)
            low = torch.einsum("bpd,kd->bkp", v, F.normalize(p["t"], dim=-1)).reshape(x.shape[0], HC, HH, HH)
            ce = F.cross_entropy(F.interpolate(low, size=lab.shape[-2:], mode="bilinear", align_corners=False), lab,
                                 ignore_index=0)
            gs = torch.autograd.grad(ce * 1.4, list(p.values()))
            with torch.no_grad():
                for t, gr in zip(p.values(), gs):
                    t -= 0.5 * gr
            losses.append(float(ce))
    return {k: v.detach() for k, v in p.items()}, losses


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", [(2, 2, 2, 1), (3, 3, 2)])
def test_graphed_engine_with_short_batches_gpu(sizes):
    """The graphed Engine runs its short batches eagerly: it trains like the eager Engine, and both like float64
    autograd (bf16 tensor-core operands: 2e-2 of the maximum, the tolerance of test_gpu_k1.py)."""
    dev = torch.device("cuda")
    loader, epochs = _head_batches(sizes, 4), 3                  # capture in epoch 2, replays in epochs 2 and 3
    init = _head_model(1)
    ref_state, ref_losses = _head_reference(init, loader, epochs)
    runs = {}
    for graph in (False, True):
        m = _head_model(1)
        eng = _head_engine(m, loader, dev, graph=graph, max_epoch=epochs)
        eng.train()
        runs[graph] = (m, [h["train_loss"] for h in eng.history], [h["train_aux_loss"] for h in eng.history], eng)
    eng = runs[True][3]
    assert eng._graph is not None and "graph" in eng._graph
    assert eng._graph["labels"].shape[0] == sizes[0]
    for (k, a), (_, b) in zip(runs[False][0].state_dict().items(), runs[True][0].state_dict().items()):
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-5), k
    for graph, (m, main, aux, _) in runs.items():
        assert len(main) == len(ref_losses) == epochs * len(sizes)
        top = max(abs(x) for x in ref_losses)
        err = max(abs(a - b) for a, b in zip(main, ref_losses)) / top
        assert err <= 2e-2, (graph, err)
        assert max(abs(a - 0.4 * b) for a, b in zip(aux, ref_losses)) / (0.4 * top) <= 2e-2
        for k, v in m.state_dict().items():
            got, ref, v0 = v.double().cpu(), ref_state[k], init.state_dict()[k].double()
            assert _rel(got, ref) <= 2e-2, (graph, k, _rel(got, ref))
            assert _rel(got - v0, ref - v0) <= 2e-2, (graph, k, "update", _rel(got - v0, ref - v0))
        print(f"graph={graph} sizes={sizes}: per-step loss {err:.2e}, weights "
              f"{max(_rel(v.double().cpu(), ref_state[k]) for k, v in m.state_dict().items()):.2e}, updates "
              f"{max(_rel(v.double().cpu() - init.state_dict()[k], ref_state[k] - init.state_dict()[k]) for k, v in m.state_dict().items()):.2e} (of max)")


_NCCL_TRAIN = dict(sizes=(4, 4, 4), seed=11, ignore=(0.0, 0.0, 0.8, 0.8))   # rank 1's images: 80 % ignored
_NCCL_EVAL = (2, 1)                                                          # all on rank 0; rank 1's shard is empty


def _nccl_eval_engine(model, loader, device):
    crit = nn.CrossEntropyLoss(ignore_index=0)                 # eval labels on the low-resolution grid
    return Engine("e", model, None, crit, aux_criterion=crit, device=device, eval_loader=loader, logger=None,
                  ignore_index=0)


def _nccl_eval_batches():
    g = torch.Generator().manual_seed(9)
    return [(dict(patches=torch.randn(b, HH * HH, 32, generator=g), label=torch.randint(0, HC, (b, HH, HH), generator=g)),
             None) for b in _NCCL_EVAL]


def _nccl_worker(rank, world, out_dir):
    dev = torch.device("cuda", rank)
    m = _head_model(rank + 1)                                  # rank 1 starts elsewhere: the broadcast must fix it
    full = _head_batches(_NCCL_TRAIN["sizes"], _NCCL_TRAIN["seed"], _NCCL_TRAIN["ignore"])
    shard = [(dict(patches=d["patches"][a:b], label=d["label"][a:b]), None)
             for d, _ in full for a, b in [dp.shard_range(d["label"].shape[0], rank, world)]]
    eng = _head_engine(m, shard, dev)
    eng.train()
    ev = _nccl_eval_engine(m, _nccl_eval_batches() if rank == 0 else [], dev)
    metrics = ev.evaluate()
    torch.save(dict(state={k: v.cpu() for k, v in m.state_dict().items()},
                    losses=[(h["train_loss"], h["train_aux_loss"]) for h in eng.history], metrics=metrics,
                    confmat=ev.last_eval_stats["confmat"].cpu(), per_image=ev.last_eval_stats["per_image"].cpu()),
               os.path.join(out_dir, f"rank{rank}.pt"))
    return "ok"


@pytest.mark.gpu
def test_two_gpu_engine_matches_single_gpu(tmp_path):
    """NCCL, unequal valid counts per rank, differently seeded replicas, an empty eval shard on rank 1: the weights and
    per-step losses are the single-GPU Engine's on the concatenated batches, and the online evaluation of the trained
    weights gives the single-GPU confusion matrix and per-image counts bit for bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    _spawn(_nccl_worker, 2, str(tmp_path), backend="nccl", timeout=600.0)
    r0, r1 = (torch.load(tmp_path / f"rank{r}.pt") for r in range(2))
    dev = torch.device("cuda", 0)
    m = _head_model(1)
    eng = _head_engine(m, _head_batches(_NCCL_TRAIN["sizes"], _NCCL_TRAIN["seed"], _NCCL_TRAIN["ignore"]), dev)
    eng.train()
    errs = {}
    for k, v in m.state_dict().items():
        assert torch.equal(r0["state"][k], r1["state"][k]), k
        errs[k] = _rel(r0["state"][k], v.cpu())
        assert errs[k] <= 1e-5, (k, errs[k])
    for (a, aa), h in zip(r0["losses"], eng.history):
        assert _rel(a, h["train_loss"]) <= 1e-5 and _rel(aa, h["train_aux_loss"]) <= 1e-5, (a, aa, h)
    for r in (r0, r1):                                         # every rank ends with the same global statistics
        assert torch.equal(r["confmat"], r0["confmat"]) and torch.equal(r["per_image"], r0["per_image"])

    # single-GPU evaluation of the weights the two ranks trained
    me = _head_model(0)
    me.load_state_dict(r0["state"])
    ev = _nccl_eval_engine(me, _nccl_eval_batches(), dev)
    met = ev.evaluate()
    assert torch.equal(r0["confmat"], ev.last_eval_stats["confmat"].cpu())
    assert torch.equal(r0["per_image"], ev.last_eval_stats["per_image"].cpu())
    assert r0["metrics"]["eval_mIOU_label"] == met["eval_mIOU_label"]
    assert r0["metrics"]["eval_mIOU_global"] == met["eval_mIOU_global"]
    assert _rel(r0["metrics"]["eval_loss"], met["eval_loss"]) <= 1e-6
    print(f"2-GPU: worst state_dict relative error {max(errs.values()):.2e}")
