"""CPU: pins oracle/restate.py against fixtures produced by the UNMODIFIED reference (oracle/make_golden.py)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import restate, synth
from oracle.digest import fixture_pair

GOLD = synth.GOLDEN_DIR
NETS = {"s_psp": "yolov5s_city_seg.yaml", "m_lab": "yolov5m_city_seg_lab.yaml", "s_bise": "yolov5s_city_seg_bise.yaml",
        "s_base": "yolov5s_city_seg_base.yaml", "m_psp": "yolov5m_city_seg.yaml"}


def relmax(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


@pytest.mark.parametrize("tag", list(NETS))
def test_forward_restatement_matches_reference(tag):
    cfg = synth.load_cfg(NETS[tag])
    sd = synth.synth_state_dict(synth.load_manifest(tag), cfg, seed=1)
    g = np.load(os.path.join(GOLD, f"net_{tag}.npz"))
    out = restate.model_forward(cfg, sd, torch.from_numpy(g["x"]), keep=(0, 4, 9, 17, 23))
    # fp32 CPU both sides; differences are only BN-fold order / oneDNN kernel choice
    assert relmax(out["z"].numpy(), g["z"]) < 2e-4
    assert relmax(*fixture_pair(g, "seg", out["seg"].numpy())) < 2e-4
    assert relmax(out["seg_lowres"].numpy(), g["seg_lowres"]) < 2e-4
    for i in range(3):
        assert out["raw"][i].shape == g[f"raw{i}"].shape
        assert relmax(out["raw"][i].numpy(), g[f"raw{i}"]) < 2e-4
    for i in (0, 4, 9, 17, 23):
        assert relmax(out["layers"][i].numpy(), g[f"layer{i}"].astype(np.float32)) < 2e-3  # taps stored as fp16


@pytest.mark.parametrize("tag", ["s_psp", "m_lab"])
def test_fp16_emulation_mode_is_close(tag):
    """The `quantised=True` graph (fp16 storage, fp32 accumulate — what the CUDA path computes) must stay within the
    north_star tolerance class of the fp32 reference: this is the budget the GPU parity tests are judged against."""
    cfg = synth.load_cfg(NETS[tag])
    sd = synth.synth_state_dict(synth.load_manifest(tag), cfg, seed=1)
    g = np.load(os.path.join(GOLD, f"net_{tag}.npz"))
    out = restate.model_forward(cfg, sd, torch.from_numpy(g["x"]), quantised=True)
    assert relmax(*fixture_pair(g, "seg", out["seg"].numpy())) < 2e-2
    assert relmax(out["raw"][0].numpy(), g["raw0"]) < 2e-2


def test_nms_restatement_bit_exact():
    g = np.load(os.path.join(GOLD, "nms_cases.npz"))
    settings = json.load(open(os.path.join(GOLD, "nms_settings.json")))
    n_checked = 0
    for name, kw in settings.items():
        for pn in ("big", "small"):
            if f"out_{name}_{pn}_0" not in g:
                continue
            outs = restate.non_max_suppression(g[f"pred_{pn}"], **kw)
            for b, o in enumerate(outs):
                ref = g[f"out_{name}_{pn}_{b}"]
                assert o.shape == ref.shape, (name, pn, b, o.shape, ref.shape)
                assert np.array_equal(o, ref), (name, pn, b)   # bit-exact rows incl. order
                n_checked += 1
    assert n_checked >= 16


def test_segpost_restatement():
    g = np.load(os.path.join(GOLD, "segpost_cases.npz"))
    for name, hw in {"x8": (128, 256), "odd": (40, 77), "same": (24, 24), "up2": (64, 128)}.items():
        am = restate.seg_postprocess(g[f"in_{name}"], hw)[0]
        ref = g[f"argmax_{name}"].astype(np.int64)
        mism = (am != ref)
        if f"up_{name}" in g:
            up = restate.bilinear_align_corners_np(g[f"in_{name}"], hw)[0]
            assert np.abs(up - g[f"up_{name}"]).max() <= 1e-5 * np.abs(g[f"up_{name}"]).max()
        # ATen's vectorised CPU kernel may contract a*b+c*d to FMA; argmax may only differ at 1-ulp near-ties
        assert mism.mean() < 1e-4, (name, mism.sum())


# ---- training losses (SURVEY.md section 8 row a13): fixtures from the unmodified reference's ComputeLoss / SegmentationLosses ----
def _loss_fixture():
    g = np.load(os.path.join(GOLD, "loss_cases.npz"))
    hyp = json.loads(bytes(g["hyp_json"]).decode())
    return g, hyp


@pytest.mark.parametrize("name", ["a", "empty", "edge"])
def test_det_loss_restatement_matches_reference(name):
    g, hyp = _loss_fixture()
    p = [torch.from_numpy(g[f"{name}_p{i}"]).requires_grad_(True) for i in range(3)]
    loss, items = restate.compute_det_loss(p, g[f"{name}_targets"], g["anchors"], hyp, nc=10)
    loss.backward()
    assert abs(float(loss.detach()) - float(g[f"{name}_loss"][0])) <= 1e-6 * abs(float(g[f"{name}_loss"][0]))
    assert np.allclose(items.numpy(), g[f"{name}_items"], rtol=1e-6, atol=1e-7)
    for i in range(3):
        assert np.abs(p[i].grad.numpy() - g[f"{name}_g{i}"]).max() <= 1e-8


@pytest.mark.parametrize("name", ["a", "empty", "edge"])
def test_det_loss_product_matches_reference(name):
    """the mask-based (synchronisation-free) product loss gives the reference's loss, loss items and gradients (fp32 tolerance 1e-5)"""
    from multiyolov5_b200.models.yolo import Model
    from multiyolov5_b200.utils.loss import ComputeLoss
    g, hyp = _loss_fixture()
    model = Model("yolov5s_city_seg.yaml")
    model.hyp, model.gr = hyp, 1.0
    assert np.allclose(model.model[-1].anchors.numpy(), g["anchors"])
    crit = ComputeLoss(model)
    p = [torch.from_numpy(g[f"{name}_p{i}"]).requires_grad_(True) for i in range(3)]
    loss, items = crit(p, torch.from_numpy(g[f"{name}_targets"]))
    loss.backward()
    assert abs(float(loss.detach()) - float(g[f"{name}_loss"][0])) <= 1e-5 * abs(float(g[f"{name}_loss"][0]))
    assert np.allclose(items.numpy(), g[f"{name}_items"], rtol=1e-5, atol=1e-6)
    for i in range(3):
        ref = g[f"{name}_g{i}"]
        assert np.abs(p[i].grad.numpy() - ref).max() <= 1e-5 * np.abs(ref).max()


def test_seg_loss_matches_reference():
    from multiyolov5_b200.utils.loss import SegmentationLosses
    g = np.load(os.path.join(GOLD, "seg_loss_cases.npz"))
    for fn in (restate.seg_ce_loss, SegmentationLosses(ignore_index=-1)):
        seg = torch.from_numpy(g["seg_logits"]).requires_grad_(True)
        loss = fn(seg, torch.from_numpy(g["seg_mask"]))
        loss.backward()
        assert abs(float(loss.detach()) - float(g["seg_loss"])) <= 1e-6
        assert np.abs(seg.grad.numpy() - g["seg_grad"]).max() <= 1e-9


# ---- pre-process (SURVEY.md section 8f rank 1): fixtures from the reference's own letterbox (cv2.resize / copyMakeBorder underneath) ----
def test_letterbox_restatement_bit_exact():
    g = np.load(os.path.join(GOLD, "letterbox_cases.npz"))
    meta = json.loads(bytes(g["meta_json"]).decode())
    assert len(meta) >= 24
    for key, m in meta.items():
        fn, sn = key.rsplit("_", 1)
        out, ratio, dwdh = restate.letterbox_np(g[f"in_{fn}"], **m["kw"])
        ref = g[f"out_{key}"]
        assert out.shape == ref.shape, (key, out.shape, ref.shape)
        assert np.array_equal(out, ref), (key, int((out != ref).sum()))          # integer arithmetic: bit exact
        assert np.allclose(ratio, m["ratio"]) and np.allclose(dwdh, m["dwdh"]), key


def test_seg_consumer_restatements_match_reference():
    g = np.load(os.path.join(GOLD, "consumer_cases.npz"))
    mask = restate.label2image_np(g["pred"], g["colormap"])[:, :, ::-1]
    assert np.array_equal(mask, g["mask_bgr"])
    assert np.array_equal(restate.label2image_np(g["pred"], g["idmap"]), g["ids"])
    assert np.array_equal(restate.add_weighted_u8(g["mask_bgr"], 0.4, g["im0"], 0.6), g["blend"])
    c, l, inter, union = restate.seg_metrics_np(g["m_out"], g["m_tgt"], 19)
    assert (c, l) == (int(g["m_correct"]), int(g["m_labeled"]))
    assert np.array_equal(inter, g["m_inter"]) and np.array_equal(union, g["m_union"])


TRAIN_NETS = {"s_psp": "yolov5s_city_seg.yaml", "s_bise": "yolov5s_city_seg_bise.yaml", "m_lab": "yolov5m_city_seg_lab.yaml",
              "s_base": "yolov5s_city_seg_base.yaml"}


@pytest.mark.parametrize("tag", list(TRAIN_NETS))
def test_train_restatement_pinned_by_reference_train_mode(tag):
    """oracle.restate.model_forward_train vs the reference's own train-mode `Model` + torch.autograd (tests/golden/train_<tag>.npz, written
    by oracle/make_golden.py gen_train): head outputs, the gradient of EVERY parameter (norm / sum / 64 samples each) and the BatchNorm
    running statistics after the forward.  This is the pin of the truth the GPU training tests are judged against."""
    from oracle.digest import grad_digest, train_probe_tensors
    cfg = synth.load_cfg(TRAIN_NETS[tag])
    sd = synth.synth_state_dict(synth.load_manifest(tag), cfg, seed=1, gain=1.0)
    g = np.load(os.path.join(GOLD, f"train_{tag}.npz"))
    x = synth.synth_image(2, 64, 96, seed=5)
    mask = None
    if "dropout_keep_bits" in g:
        shp = tuple(int(v) for v in g["dropout_shape"])
        mask = torch.from_numpy(np.unpackbits(g["dropout_keep_bits"])[:int(np.prod(shp))].reshape(shp).astype(np.float32))
    sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k and "anchor" not in k else v.clone())
           for k, v in sd.items()}
    new_running = {}
    raws, seg = restate.model_forward_train(cfg, sdg, x, mask, new_running=new_running)
    segs = list(seg) if isinstance(seg, (list, tuple)) else [seg]
    Rs, Ss = train_probe_tensors([tuple(r.shape) for r in raws], [tuple(s.shape) for s in segs])
    loss = sum((r * R).sum() for r, R in zip(raws, Rs)) + sum((s * S).sum() for s, S in zip(segs, Ss))
    loss.backward()
    for i, r in enumerate(raws):
        assert relmax(r.detach().numpy(), g[f"raw{i}"]) < 1e-4, (i, relmax(r.detach().numpy(), g[f"raw{i}"]))
    for k, s in enumerate(segs):
        assert relmax(s.detach()[:, :, ::3, ::3].numpy(), g[f"seg{k}_sub"]) < 1e-4
    assert abs(float(loss) - float(g["loss"])) < 1e-3 * max(1.0, abs(float(g["loss"])))
    # every gradient the reference produced exists here, under the same name, with the same digest
    names = [str(n) for n in g["grad_names"]]
    dig = g["grad_digest"]
    norm_errs = []
    for n, d in zip(names, dig):
        assert sdg[n].grad is not None, n
        mine = grad_digest(sdg[n].grad)
        scale = max(d[0] / np.sqrt(sdg[n].numel()), 1e-12)       # RMS magnitude of the tensor
        err_norm = abs(mine[0] - d[0]) / max(d[0], 1e-12)
        err_samples = float(np.abs(mine[2:] - d[2:]).max() / scale)
        norm_errs.append(err_norm)
        assert err_norm < 2e-3, (n, mine[0], d[0])
        # single entries relative to the tensor's RMS.  The Base head's C3SPP max-pools an 8x12 map with 9x9 / 13x13 windows: two candidates
        # that tie to 1e-7 route the whole window gradient to a different pixel (same d gamma / d beta, different d W upstream) - measured
        # 1e-2 Frobenius on those tensors between the reference and this restatement, both fp32 torch
        assert err_samples < (0.15 if tag == "s_base" else 2e-2), (n, err_samples)
    assert float(np.median(norm_errs)) < (3e-3 if tag == "s_base" else 1e-4), float(np.median(norm_errs))
    assert len(names) == sum(1 for v in sdg.values() if v.requires_grad and v.grad is not None)
    # running statistics (momentum 0.03, unbiased variance)
    off = 0
    for n in [str(v) for v in g["bn_names"]]:
        rm, rv = new_running[n]
        c = rm.numel()
        assert np.allclose(rm.numpy(), g["bn_mean"][off:off + c], rtol=1e-4, atol=1e-6), n
        assert np.allclose(rv.numpy(), g["bn_var"][off:off + c], rtol=1e-4, atol=1e-6), n
        off += c
    assert off == g["bn_mean"].size


BIG = {"s_psp_256x512": ("s_psp", "yolov5s_city_seg.yaml"), "m_lab_256x512": ("m_lab", "yolov5m_city_seg_lab.yaml")}


@pytest.mark.parametrize("name", list(BIG))
def test_forward_restatement_matches_reference_at_tensor_core_sizes(name):
    """the tcgen05-sized reference fixtures (netbig_*.npz) also pin the restatement (fp32 CPU both sides)"""
    tag, yml = BIG[name]
    cfg = synth.load_cfg(yml)
    sd = synth.synth_state_dict(synth.load_manifest(tag), cfg, seed=1)
    g = np.load(os.path.join(GOLD, f"netbig_{name}.npz"))
    B, H, W = [int(v) for v in g["shape"]]
    x = synth.synth_image(B, H, W, seed=int(g["seed"]))
    assert abs(float(x.double().sum()) - float(g["x_sum"])) < 1e-6 * float(g["x_sum"])
    out = restate.model_forward(cfg, sd, x, keep=(9, 23))
    assert relmax(*fixture_pair(g, "z", out["z"].numpy())) < 2e-4
    assert relmax(out["seg_lowres"].numpy(), g["seg_lowres"]) < 2e-4
    for i in range(3):
        assert relmax(*fixture_pair(g, f"raw{i}", out["raw"][i].numpy())) < 1e-3      # stored as fp16
    for i in (9, 23):
        assert relmax(*fixture_pair(g, f"layer{i}", out["layers"][i].numpy())) < 2e-3
    agree = float((out["seg"].argmax(1).numpy() == g["seg_argmax"]).mean())
    assert agree > 0.9999, agree
