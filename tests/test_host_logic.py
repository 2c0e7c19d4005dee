"""Host-side mirror of the reference interface, CPU-checkable parts."""
import os

import pytest
import torch

from oracle import head_oracle as O
from lc2is_b200 import metrics, synthetic
from lc2is_b200.model import TextToPatch, AuxiliaryLoss, ContrastiveLoss, NPairLoss
from lc2is_b200.model.decoder import DecoderLayer, DecoderBlock, PromptLayer, PromptDecoder


def test_text_to_patch_matches_reference(golden_dir):
    g = torch.load(os.path.join(golden_dir, "text_patch.pt"))
    m = TextToPatch(img_in=48, text_in=32, out=64)
    m.load_state_dict(g["state"])                                # reference parameter names load
    tf, vf = m(g["img"], g["text"])                              # text first (text_patch.py:18)
    assert torch.equal(tf, g["t_feature"]) and torch.equal(vf, g["v_feature"])
    assert sum(p.numel() for p in TextToPatch(768, 512, 512).parameters()) == 656384


def test_miou_helpers_match_oracle():
    g = torch.Generator().manual_seed(3)
    cm = torch.randint(0, 50, (7, 7), generator=g)
    cm[:, 5] = 0; cm[5, :] = 0                                   # an absent class
    for ign in (0, 3, None):
        a = metrics.miou_from_confmat(cm, ign).item()
        b = O.jaccard_macro(cm, ign).item()
        assert abs(a - b) < 1e-7
        assert abs(metrics.pixel_accuracy_from_confmat(cm, ign).item() - O.pixel_accuracy(cm, ign)) < 1e-12


def test_per_image_miou_matches_oracle():
    g = torch.Generator().manual_seed(4)
    C = 6
    pred = torch.randint(0, C, (3, 10, 10), generator=g)
    lab = torch.randint(0, C, (3, 10, 10), generator=g)
    lab[1][lab[1] == 4] = 2                                       # class 4 absent from image 1's label
    per = torch.zeros(3, 3, C, dtype=torch.int64)
    ref = []
    for n in range(3):
        cm = O.confusion_matrix(pred[n], lab[n], C)
        per[n, 0] = torch.diag(cm); per[n, 1] = cm.sum(1); per[n, 2] = cm.sum(0)
        ref.append(O.per_image_miou_from_cm(cm, lab[n], 0))
    got = metrics._per_image_miou(per, 0)
    torch.testing.assert_close(got, torch.cat(ref), rtol=0, atol=1e-7)


def test_auxiliary_loss_rejects_unsupported_options():
    with pytest.raises(NotImplementedError):
        AuxiliaryLoss(weight=torch.ones(3))
    with pytest.raises(NotImplementedError):
        AuxiliaryLoss(label_smoothing=0.1)
    with pytest.raises(NotImplementedError):
        AuxiliaryLoss(reduction="none")
    assert AuxiliaryLoss(ignore_index=0).ignore_index == 0


def test_passthrough_losses_run():
    r = NPairLoss()(torch.rand(4, 8), torch.rand(3, 8), torch.rand(5, 8))
    assert r.shape == ()


def test_contrastive_loss_surface():
    from lc2is_b200._lib import Lc2isError
    with pytest.raises(NotImplementedError):
        ContrastiveLoss(label_smoothing=0.1)
    with pytest.raises(NotImplementedError):
        ContrastiveLoss(reduction="sum")
    with pytest.raises(RuntimeError, match="floating point target"):     # same as the reference's criterion
        ContrastiveLoss(ignore_index=0)(torch.randn(2, 16, 151), torch.randint(0, 4, (2, 4, 4)))
    crit = ContrastiveLoss()
    assert crit.criterion.ignore_index == -100
    with pytest.raises(ValueError):                      # C != 151: the reference's one-hot target cannot match
        crit(torch.randn(2, 16, 150), torch.randint(0, 4, (2, 4, 4)))
    with pytest.raises(ValueError):                      # labels at another resolution
        crit(torch.randn(2, 16, 151), torch.randint(0, 4, (2, 8, 8)))
    with pytest.raises(Lc2isError):                      # no CPU path
        crit(torch.randn(2, 16, 151), torch.randint(0, 4, (2, 4, 4)))


def test_decoder_surface():
    layer = DecoderLayer(d_model=32, d_kv=16, nhead=4, dim_feedforward=64, batch_first=True, norm_first=True)
    blk = DecoderBlock(layer, num_layers=1)
    y = blk(tgt=torch.randn(2, 5, 32), memory=torch.randn(2, 3, 16))
    assert y.shape == (2, 5, 32)
    p = PromptDecoder(PromptLayer(d_model=32, d_kv=16, nhead=4, dim_feedforward=64, batch_first=True), 1)
    assert p(torch.randn(2, 5, 32), torch.randn(2, 3, 16)).shape == (2, 5, 32)


def test_synthetic_inputs_are_seeded():
    a = synthetic.make_labels(2, 64, 64, 151)
    b = synthetic.make_labels(2, 64, 64, 151)
    assert torch.equal(a, b) and a.dtype == torch.int64 and int(a.max()) < 151 and int(a.min()) >= 0
    assert synthetic.make_prototypes(150).shape == (150, 512)
    assert torch.equal(synthetic.make_prototypes(150), synthetic.load_prototypes()[1:])
    assert synthetic.make_prototypes(847).shape == (847, 512)
    d = synthetic.make_dyadic_logits(1, 5, 4, 4)
    assert torch.equal(d * 256, (d * 256).round())


def test_host_label_packing_matches_device_encoding():
    """lc2is_pack_labels_host (HOST code, worker pool + AVX2).  C > 254: int64 -> uint16 class id, bit 15 = ignore_index,
    0xFFFF = not a class id.  C <= 254: one byte, 0xFE = ignore_index, 0xFF = not a class id.  Ragged lengths exercise
    the scalar tail."""
    import torch
    from lc2is_b200 import _lib
    g = torch.Generator().manual_seed(9)
    for n, C, ign in ((1, 5, 0), (17, 151, 0), (100003, 150, -100), (4 * 512 * 512, 847, 3), (70001, 254, 253),
                      (33, 255, 0)):
        lab = torch.randint(-3, C + 4, (n,), generator=g)
        lab[:: max(1, n // 7)] = ign
        if n > 3:
            lab[1], lab[2], lab[3] = 2 ** 40, -2 ** 40, 65535
        nb = _lib.lib.lc2is_host_label_bytes(C)
        assert nb == (1 if C <= 254 else 2)
        inr = (lab >= 0) & (lab < C)
        if nb == 2:
            out = torch.full((n + 8,), 7, dtype=torch.uint16)
            ref = torch.where(inr, torch.where(lab == ign, lab | 0x8000, lab), torch.full_like(lab, 0xFFFF))
        else:
            out = torch.full((n + 8,), 7, dtype=torch.uint8)
            ref = torch.where(inr, torch.where(lab == ign, torch.full_like(lab, 0xFE), lab), torch.full_like(lab, 0xFF))
        _lib.check(_lib.lib.lc2is_pack_labels_host(lab.data_ptr(), n, C, ign, out.data_ptr()), "pack")
        assert torch.equal(out[:n].to(torch.int64), ref)
        assert bool((out[n:] == 7).all())                     # nothing written past the end
        # the asynchronous form writes the same bytes
        out2 = torch.full_like(out, 7)
        import ctypes
        hd = ctypes.c_void_p()
        _lib.check(_lib.lib.lc2is_pack_labels_host_begin(lab.data_ptr(), n, C, ign, out2.data_ptr(), ctypes.byref(hd)), "begin")
        _lib.check(_lib.lib.lc2is_pack_labels_host_end(hd), "end")
        assert torch.equal(out, out2)


def test_host_label_packing_avx2_path_in_a_subprocess():
    """The AVX-512 / AVX2 choice is made once per process: run the same encoding check with AVX-512 switched off."""
    import os, subprocess, sys
    code = (
        "import torch\n"
        "from lc2is_b200 import _lib\n"
        "g = torch.Generator().manual_seed(3)\n"
        "for n, C, ign in ((100003, 150, 0), (65536, 847, 3), (33, 254, 253)):\n"
        "    lab = torch.randint(-3, C + 4, (n,), generator=g); lab[::5] = ign\n"
        "    nb = _lib.lib.lc2is_host_label_bytes(C)\n"
        "    inr = (lab >= 0) & (lab < C)\n"
        "    if nb == 2:\n"
        "        out = torch.zeros(n, dtype=torch.uint16); ref = torch.where(inr, torch.where(lab == ign, lab | 0x8000, lab), torch.full_like(lab, 0xFFFF))\n"
        "    else:\n"
        "        out = torch.zeros(n, dtype=torch.uint8); ref = torch.where(inr, torch.where(lab == ign, torch.full_like(lab, 0xFE), lab), torch.full_like(lab, 0xFF))\n"
        "    _lib.check(_lib.lib.lc2is_pack_labels_host(lab.data_ptr(), n, C, ign, out.data_ptr()), 'pack')\n"
        "    assert torch.equal(out.to(torch.int64), ref), (n, C)\n"
        "print('ok')\n")
    env = dict(os.environ, LC2IS_NO_AVX512="1", LC2IS_PACK_THREADS="3")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=root, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]


def test_label_route_selection_rule():
    """HostStep.pick_raw_images: all label maps packed on a fast host, a growing share sent as int64 as the host gets
    slower, everything raw when packing is hopeless (numbers of the bench shape: B=16, 512^2 labels, 16.8 MB of V)."""
    from lc2is_b200.step import HostStep
    B, HW, v = 16, 512 * 512, 16 * 1024 * 512 * 2
    pick = lambda pack_ms, gbs: HostStep.pick_raw_images(B, v, HW, HW * 8, pack_ms * 1e-3 / B, gbs * 1e9)
    assert pick(0.30, 55) == 0 and pick(0.42, 55) == 0             # packing at or below the copy time: stay all-packed
    picks = [pick(ms, 55) for ms in (0.6, 1.0, 2.0, 5.0, 50.0)]
    assert picks == sorted(picks) and picks[0] >= 1 and picks[-1] >= 15
    assert pick(1.0, 10) <= pick(1.0, 55)                           # a slow link keeps more of the packing on the host
    for ms, gbs in ((0.6, 55), (2.2, 52), (1.0, 20)):
        r = pick(ms, gbs)
        t = lambda k: max(ms * 1e-3 / B * (B - k), (v + (B - k) * HW + k * HW * 8) / (gbs * 1e9))
        assert t(r) <= 1.05 * min(t(k) for k in range(B + 1)) + 1e-12


def test_host_label_packing_property():
    """Property test (hypothesis): any int64 label vector, class count and ignore_index pack to the documented codes,
    for the one-byte and the two-byte host form alike, whatever the length / alignment of the slice."""
    hyp = pytest.importorskip("hypothesis")
    st = pytest.importorskip("hypothesis.strategies")
    from lc2is_b200 import _lib
    special = [0, 1, -1, 253, 254, 255, 256, 32766, 32767, 65535, 65536, 2 ** 31, -2 ** 31, 2 ** 62, -2 ** 62]

    @hyp.settings(max_examples=150, deadline=None)
    @hyp.given(st.integers(1, 600), st.integers(1, 300), st.sampled_from([-100, -1, 0, 3, 253, 299]),
               st.integers(0, 7), st.randoms(use_true_random=False))
    def check(C, n, ign, off, rnd):
        vals = [rnd.choice(special) if rnd.random() < 0.2 else rnd.randrange(-2, C + 2) for _ in range(n)]
        lab = torch.tensor([0] * off + vals, dtype=torch.int64)[off:]          # misaligned view of the source
        nb = _lib.lib.lc2is_host_label_bytes(C)
        out = torch.full((n + 16,), 9, dtype=torch.uint8 if nb == 1 else torch.uint16)
        _lib.check(_lib.lib.lc2is_pack_labels_host(lab.data_ptr(), n, C, ign, out.data_ptr()), "pack")
        inr = (lab >= 0) & (lab < C)
        if nb == 1:
            ref = torch.where(inr, torch.where(lab == ign, torch.full_like(lab, 0xFE), lab), torch.full_like(lab, 0xFF))
        else:
            ref = torch.where(inr, torch.where(lab == ign, lab | 0x8000, lab), torch.full_like(lab, 0xFFFF))
        assert torch.equal(out[:n].to(torch.int64), ref)
        assert bool((out[n:] == 9).all())

    check()


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU oracle timed on the host cores) runs without a GPU and prints ONE JSON line
    with the keys the driver reads."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0"], cwd=root,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] == "port"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and "workload" in line["config"]


def test_bench_write_outputs_within_budget_and_repeatable(tmp_path):
    """bench.py --dump-outputs: float arrays as float32, integer arrays as float64; arrays within their share of the
    byte budget are written whole, larger ones as a seeded sample of their elements; the same files on every call."""
    import numpy as np
    import bench
    g = torch.Generator().manual_seed(5)
    arrays = {"loss": torch.tensor([1.5]), "n_valid": torch.tensor([7], dtype=torch.int64),
              "confmat": torch.randint(0, 1 << 40, (9, 9), generator=g), "logits": torch.randn(40, 30, generator=g),
              "grad_v": torch.randn(300, 500, generator=g).bfloat16()}
    budget = 200_000
    for d in ("a", "b"):
        bench.write_outputs(arrays, str(tmp_path / d), budget=budget)
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in arrays)
    got = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in arrays}
    assert sum(x.nbytes for x in got.values()) <= budget
    assert {n: x.dtype for n, x in got.items()} == {"loss": np.float32, "n_valid": np.float64, "confmat": np.float64,
                                                     "logits": np.float32, "grad_v": np.float32}
    for n in ("loss", "n_valid", "confmat", "logits"):
        assert np.array_equal(got[n], (arrays[n].float() if arrays[n].is_floating_point() else arrays[n].double()).numpy())
    gv = got["grad_v"]
    assert gv.ndim == 1 and 0.9 * budget / 2 / 4 < gv.size < 300 * 500
    assert np.isin(gv, arrays["grad_v"].float().numpy()).all()
    for n in arrays:
        assert np.array_equal(got[n], np.load(tmp_path / "b" / (n + ".npy")))


def test_ftn_decoder_mirrors_run_and_keep_the_reference_parameter_names():
    """decoder.py:36-134 mirrors (pass-through PyTorch, upstream of the head): they run on torch >= 2 (the reference's
    `_sa_block` override lacks `is_causal` there) and name their parameters like the reference."""
    import torch
    from lc2is_b200.model.decoder import FTNBlock, FTNDecoder, SRTransformerDecoder
    torch.manual_seed(0)
    dec = FTNDecoder([32, 64, 128, 256], 64, dropout=0.0).eval()
    vis = [torch.randn(2, 16 * 16, 32), torch.randn(2, 8 * 8, 64), torch.randn(2, 4 * 4, 128), torch.randn(2, 2 * 2, 256)]
    out = dec(vis, torch.randn(2, 5, 64))
    assert out.shape == (2, 256, 64) and torch.isfinite(out).all()
    names = set(dec.state_dict())
    for n in ("linear_stage_2.weight", "linear_stage_3.weight", "linear2_stage_1.weight", "linear2_stage_4.bias",
              "attention_stage_4.2.attention_block.sr.weight", "attention_stage_2.0.attention_block.norm.weight",
              "attention_stage_3.1.attention_block.self_attn.in_proj_weight"):
        assert n in names, n
    blk = FTNBlock(SRTransformerDecoder(d_model=64, nhead=8, sr_ratio=2, dropout=0.0, batch_first=True)).eval()
    assert blk(tgt=torch.randn(1, 16, 64), memory=torch.randn(1, 3, 64)).shape == (1, 64, 64)


def test_ragged_descriptor_table():
    """The descriptor table of lc2is_argmax_confmat_ragged (host logic): element offsets are the running sum of H*W, first
    tiles the running sum of lc2is_ragged_tiles (64 x 32 pixel tiles), images without pixels own no tile."""
    from lc2is_b200 import ops
    from lc2is_b200._lib import lib
    sizes = [(64, 64), (1, 1), (33, 65), (0, 5), (100, 7)]
    desc, n_tiles, n_elem = ops.ragged_descriptors(sizes)
    assert desc.shape == (5, 4) and desc.dtype == torch.int64
    tiles = [2 * 1, 1, 2 * 2, 0, 4 * 1]
    assert [int(lib.lc2is_ragged_tiles(h, w)) for h, w in sizes] == tiles
    assert desc[:, 0].tolist() == [0, 4096, 4097, 4097 + 33 * 65, 4097 + 33 * 65]
    assert desc[:, 3].tolist() == [0, 2, 3, 7, 7] and n_tiles == 11 and n_elem == 4097 + 33 * 65 + 700
    assert desc[:, 1:3].tolist() == [list(s) for s in sizes]
