"""Whole-step entry points (lc2is_head_step_host from HOST buffers; HeadStep on device buffers) against
the CPU oracle, and HeadStep == the op-by-op path."""
import pytest
import torch

from oracle import head_oracle as O
from lc2is_b200 import metrics, ops, synthetic
from lc2is_b200.step import HeadStep, HostStep

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _inputs(B, h, H, C):
    v = synthetic.make_patch_embeddings(B, h * h, 512, dtype=torch.bfloat16)
    t = synthetic.make_prototypes(C, 512)
    labels = synthetic.make_labels(B, H, H, C, block=8, ignore_frac=0.1)
    return v, t, labels


@pytest.mark.parametrize("pipelined", [False, True])
@pytest.mark.parametrize("B,h,H,C,raw", [(5, 8, 128, 151, 0), (5, 8, 128, 151, 2), (5, 8, 128, 151, 5), (4, 32, 128, 150, 0),
                                         (1, 8, 32, 19, 0), (4, 16, 128, 151, 1), (3, 8, 128, 300, 1)])
def test_host_step_matches_oracle(pipelined, B, h, H, C, raw):
    """x16 (fused kernel), x8 (separate split kernels), x4 (generic) geometries; `raw` of the label maps cross PCIe
    as int64 and are packed on the device, the others are narrowed on the host (1 byte per label, 2 for C = 300)."""
    v, t, labels = _inputs(B, h, H, C)
    ref = O.head_step(v.float(), t, labels, ignore_index=0, n_cls=C)
    hs = HostStep(B, h, h, H, H, C, ignore_index=0, pipelined=pipelined, raw_images=raw)
    for _ in range(2):                                    # twice: workspace reuse across calls
        hs(v.pin_memory(), t.pin_memory(), labels.pin_memory())
    assert int(hs.out_n_valid) == int((labels != 0).sum())
    assert abs(float(hs.out_loss) - float(ref["loss"])) <= 1e-4 * float(ref["loss"])
    # confusion matrix: exact against the oracle fed with the kernel-precision logits is covered in
    # test_gpu_k3; here: same totals and (bf16 logits vs fp32 oracle) nearly the same matrix
    cm = hs.out_confmat
    assert int(cm.sum()) == B * H * H
    assert torch.equal(cm.sum(1), torch.bincount(labels.flatten(), minlength=C))
    assert int((cm - ref["confmat"]).abs().sum()) <= 0.02 * B * H * H


def test_head_step_device_matches_oracle_and_host_step():
    B, h, H, C = 4, 32, 128, 151
    v, t, labels = _inputs(B, h, H, C)
    ref = O.head_step(v.float(), t, labels, ignore_index=0, n_cls=C)
    step = HeadStep(B, h, h, H, H, C, ignore_index=0)
    step(v.to(DEV), t.to(DEV), labels.to(DEV))
    torch.cuda.synchronize()
    assert abs(float(step.loss) - float(ref["loss"])) <= 1e-4 * float(ref["loss"])
    assert int(step.n_valid) == int((labels != 0).sum())
    gt = step.grad_t[0].cpu()
    assert float((gt - ref["grad_t"]).abs().max() / ref["grad_t"].abs().max()) < 3e-2
    gv = step.grad_v.float().cpu()
    assert float((gv - ref["grad_v"]).abs().max() / ref["grad_v"].abs().max()) < 3e-2
    hs = HostStep(B, h, h, H, H, C, ignore_index=0)
    hs(v.pin_memory(), t.pin_memory(), labels.pin_memory())
    assert torch.equal(hs.out_confmat, step.confmat.cpu())
    assert abs(float(hs.out_loss) - float(step.loss)) <= 2e-6 * float(step.loss)
    assert abs(float(metrics.miou_from_confmat(step.confmat, 0)) - float(O.jaccard_macro(step.confmat.cpu(), 0))) < 1e-7


@pytest.mark.parametrize("raw", [0, 1, 3])
def test_submit_wait_pipeline_matches_blocking_call(raw):
    """Two steps in flight (lc2is_head_step_host_submit / _wait) over alternating batches give, step by step,
    exactly the results of the blocking call; host-side label packing on and off agree bit for bit."""
    B, h, H, C = 4, 8, 128, 151
    batches = []
    for k in range(3):
        v = synthetic.make_patch_embeddings(B, h * h, 512, seed=100 + k).pin_memory()
        lab = synthetic.make_labels(B, H, H, C, seed=100 + k, block=8, ignore_frac=0.1)
        lab[0, 0, :4] = torch.tensor([-100, C, 255, 2 ** 40])          # not class ids: skipped everywhere
        batches.append((v, lab.pin_memory()))
    t = synthetic.make_prototypes(C, 512).pin_memory()
    ref = []
    blocking = HostStep(B, h, h, H, H, C, ignore_index=0, host_pack=False)
    for v, lab in batches:
        blocking(v, t, lab)
        ref.append((float(blocking.out_loss), int(blocking.out_n_valid), blocking.out_confmat.clone()))
    hs = HostStep(B, h, h, H, H, C, ignore_index=0, depth=2, raw_images=raw)
    assert hs.host_pack and hs.n_raw == raw
    got = []
    seq = [0, 1, 2, 0, 1, 2, 1]
    hs.submit(batches[seq[0]][0], t, batches[seq[0]][1])
    for j, k in enumerate(seq[1:], start=1):
        hs.submit(batches[k][0], t, batches[k][1])
        if j + 1 < len(seq) and j % 2 == 0:                    # every other batch: labels packed in the background
            hs.prefetch(batches[seq[j + 1]][1])
        l, nv, cm = hs.wait()
        got.append((float(l), int(nv), cm.clone()))
    l, nv, cm = hs.wait()
    got.append((float(l), int(nv), cm.clone()))
    for k, g in zip(seq, got):
        assert g[1] == ref[k][1] and torch.equal(g[2], ref[k][2])
        assert abs(g[0] - ref[k][0]) <= 2e-6 * abs(ref[k][0])


def test_config5_open_vocab_shape_against_eager_torch():
    """BASELINE config 5 shape (1024^2 input = 64x64 patch grid, C=847 open-vocabulary prototypes), one image per
    step: HeadStep (K1 with N-tiling, split K2 / K3 strip kernels - the fused kernel does not fit 847 classes)
    against eager torch on the same device (the CPU oracle would need 3.5 GB for the upsampled map)."""
    import torch.nn.functional as F
    B, h, H, C = 1, 64, 1024, 847
    v, t, labels = _inputs(B, h, H, C)
    step = HeadStep(B, h, h, H, H, C, ignore_index=0)
    assert step.split and not step.fused
    vd, td, ld = v.to(DEV), t.to(DEV), labels.to(DEV)
    step(vd, td, ld)
    torch.cuda.synchronize()
    # eager reference on the kernel's own logits (bf16-operand GEMM) for loss / confusion matrix ...
    low = step.logits.detach().clone().requires_grad_(True)
    up = F.interpolate(low, mode="bilinear", size=H)
    ref_loss = F.cross_entropy(up, ld, ignore_index=0)
    ref_loss.backward()
    assert abs(float(step.loss) - float(ref_loss)) <= 3e-6 * float(ref_loss)
    nv = int((ld != 0).sum())
    assert int(step.n_valid) == nv
    g = step.grad_low / nv
    assert float((g - low.grad).abs().max()) <= 2e-5 * float(low.grad.abs().max())
    pred = up.detach().argmax(1)
    cm_ref = torch.bincount((ld * C + pred).flatten(), minlength=C * C).view(C, C)
    # fp32 evaluation order may flip near-ties: totals exact, matrix equal up to a handful of pixels
    assert int(step.confmat.sum()) == B * H * H
    assert torch.equal(step.confmat.sum(1), torch.bincount(ld.flatten(), minlength=C))
    assert int((step.confmat - cm_ref).abs().sum()) <= 2e-5 * B * H * H
    # ... and the fp32 reference logits for K1 (bf16 operands: 4e-3 absolute, SURVEY 8c)
    ref_low = O.cosine_logits(v.float(), t, hw_shape=(h, h))
    assert float((step.logits.cpu() - ref_low).abs().max()) < 4e-3


def test_new_entries_reject_unsupported_geometries_loudly():
    """The split / fused / packed entries are specialised (power-of-two scales); anything else must come back as an
    error code with a message - never a silent fallback."""
    from lc2is_b200 import _lib
    lib = _lib.lib
    assert lib.lc2is_ce_split_supported(32, 32, 512, 512) == 1 and lib.lc2is_ce_split_supported(16, 16, 128, 128) == 1
    assert lib.lc2is_ce_split_supported(32, 32, 128, 128) == 0 and lib.lc2is_ce_split_supported(13, 13, 37, 37) == 0
    assert lib.lc2is_ce_argmax_fused_supported(150, 32, 32, 512, 512) == 1
    assert lib.lc2is_ce_argmax_fused_supported(847, 64, 64, 1024, 1024) == 0       # tap tile too large
    assert lib.lc2is_ce_argmax_fused_supported(150, 16, 16, 128, 128) == 0         # x8
    low = torch.zeros(1, 5, 8, 8, device=DEV)
    lab = torch.zeros(1, 32, 32, dtype=torch.int64, device=DEV)                    # x4
    pk = torch.zeros(1, 32, 32, dtype=torch.uint16, device=DEV)
    ls = torch.zeros(1, dtype=torch.float64, device=DEV)
    cm = torch.zeros(5, 5, dtype=torch.int64, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    assert lib.lc2is_upsample_ce_packed(low.data_ptr(), pk.data_ptr(), 1, 5, 8, 8, 32, 32, ls.data_ptr(), None, st) == -4
    assert "scale" in _lib.last_error()
    assert lib.lc2is_ce_argmax_fused_packed(low.data_ptr(), pk.data_ptr(), 1, 5, 8, 8, 32, 32, ls.data_ptr(), None, 1, None,
                                            cm.data_ptr(), None, None, st) == -4
    assert lib.lc2is_argmax_confmat_lowres_packed(low.data_ptr(), 1, 5, 8, 8, 32, 32, pk.data_ptr(), cm.data_ptr(), None,
                                                  None, st) == -4
    assert lib.lc2is_pack_labels(lab.data_ptr(), 7, 5, 0, pk.data_ptr(), None, st) == -2          # n % 8
    assert lib.lc2is_upsample_ce_packed(None, pk.data_ptr(), 1, 5, 2, 2, 32, 32, ls.data_ptr(), None, st) == -1
    # the x4 geometry still works end to end through the general entries (HeadStep picks them itself)
    step = HeadStep(1, 8, 8, 32, 32, 5, ignore_index=0)
    assert not step.split and not step.fused
    v = synthetic.make_patch_embeddings(1, 64, 512).to(DEV)
    step(v, synthetic.make_prototypes(5, 512).to(DEV), torch.randint(0, 5, (1, 32, 32), device=DEV))
    torch.cuda.synchronize()
    assert torch.isfinite(step.loss).all() and int(step.confmat.sum()) == 32 * 32


@pytest.mark.parametrize("C,ign", [(150, 0), (254, 253), (7, -100)])
def test_one_byte_host_labels_expand_to_the_device_packing(C, ign):
    """lc2is_pack_labels_host (1 byte per label for C <= 254) + lc2is_expand_labels == lc2is_pack_labels on the int64
    map, bit for bit, including labels outside [0,C) and the counted-pixel total."""
    from lc2is_b200 import _lib
    g = torch.Generator().manual_seed(5)
    lab = torch.randint(-2, C + 3, (2, 64, 64), generator=g)
    lab[0, :8] = ign
    assert _lib.lib.lc2is_host_label_bytes(C) == 1
    h8 = torch.empty(lab.shape, dtype=torch.uint8).pin_memory()
    _lib.check(_lib.lib.lc2is_pack_labels_host(lab.data_ptr(), lab.numel(), C, ign, h8.data_ptr()), "pack")
    nv = torch.zeros(1, dtype=torch.int64, device=DEV)
    got = ops.expand_labels(h8.to(DEV), C, ign, nv)
    want, nv_ref = ops.pack_labels(lab.to(DEV), C, ign)
    assert torch.equal(got.cpu().view(torch.int16), want.cpu().view(torch.int16))
    assert int(nv) == int(nv_ref) == int(((lab >= 0) & (lab < C) & (lab != ign)).sum())


def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """`bench.py --steps 2 --dump-outputs DIR`: two timed steps (the confusion matrix of the pass counts two batches)
    and the dumped loss / n_valid / logits / gradients are those of HeadStep on the second input set."""
    import json, os, subprocess, sys
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, "bench.py", "--steps", "2", "--warmup", "1", "--no-e2e", "--no-secondary",
                        "--no-cpu-baseline", "--dump-outputs", str(out)], cwd=root, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    B, h, H, C = 16, 32, 512, 150
    assert line["steps"] == 2 and line["check"]["confmat_total"] == 2 * B * H * H
    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert set(got) == {"loss", "n_valid", "logits", "confmat", "grad_v", "grad_t"}
    assert sum(x.nbytes for x in got.values()) <= 64 * 10 ** 6
    assert got["confmat"].dtype == np.float64 and got["confmat"].sum() == 2 * B * H * H

    seed = synthetic.SEED + 97 * 1                              # bench.py's input set of timed step 1
    v = synthetic.make_patch_embeddings(B, h * h, 512, seed=seed).to(DEV)
    lab = synthetic.make_labels(B, H, H, C, seed=seed, ignore_frac=0.1).to(DEV)
    step = HeadStep(B, h, h, H, H, C, ignore_index=0)
    step(v, synthetic.make_prototypes(C, 512).to(DEV), lab)
    torch.cuda.synchronize()
    assert got["n_valid"].tolist() == [int(step.n_valid)]
    assert abs(float(got["loss"][0]) - float(step.loss)) <= 1e-5 * abs(float(step.loss))
    torch.testing.assert_close(torch.from_numpy(got["logits"]), step.logits.cpu(), rtol=1e-5, atol=1e-6)
    for name, ref in (("grad_t", step.grad_t), ("grad_v", step.grad_v)):
        ref = ref.float().cpu()
        assert got[name].shape == tuple(ref.shape)
        assert float((torch.from_numpy(got[name]) - ref).abs().max()) <= 1e-2 * float(ref.abs().max()), name


def test_default_host_step_calibrates_the_label_split():
    """Without `raw_images` the step measures the host's packing rate and the H2D rate and picks how many label maps
    cross as int64; whatever it picks, the results are those of the all-raw step."""
    B, h, H, C = 4, 8, 128, 151
    v, t, labels = _inputs(B, h, H, C)
    hs = HostStep(B, h, h, H, H, C, ignore_index=0)
    assert 0 <= hs.n_raw <= B and hs.calibration["pack_ms"] > 0 and hs.calibration["h2d_gbs"] > 1
    ref = HostStep(B, h, h, H, H, C, ignore_index=0, host_pack=False)
    for s_ in (hs, ref):
        s_(v.pin_memory(), t.pin_memory(), labels.pin_memory())
    assert torch.equal(hs.out_confmat, ref.out_confmat) and int(hs.out_n_valid) == int(ref.out_n_valid)
    assert abs(float(hs.out_loss) - float(ref.out_loss)) <= 2e-6 * float(ref.out_loss)
