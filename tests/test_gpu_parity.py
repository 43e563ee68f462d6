"""GPU parity at the configurations that matter (VERDICT round 1, items 1a-1d):

  * `Model.forward` against fixtures produced by the UNMODIFIED reference at sizes where every conv runs on the tcgen05 kernel
    (tests/golden/netbig_*.npz: s/PSP and m/Lab at 256x512, s/PSP at 512x1024), per-output tolerances, box error in PIXELS;
  * a yardstick for what fp16 activation storage costs: the same graph through torch's own fp16 CUDA kernels - the reference's GPU
    configuration, detect.py:96-103 - measured against the same fp32 fixtures; ours must not be further away than that;
  * end to end at BASELINE.json configs[1] (batch 16 x 512 x 1024, half mode): class-id agreement with the fp32 oracle and equality of the
    detection sets modulo boxes whose score / IoU lies within a stated epsilon of a threshold (SURVEY.md section 7 (ii)).
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import restate, synth
from oracle.digest import fixture_pair

pytestmark = pytest.mark.gpu
BIG = {"s_psp_256x512": ("s_psp", "yolov5s_city_seg.yaml"), "m_lab_256x512": ("m_lab", "yolov5m_city_seg_lab.yaml"),
       "s_psp_512x1024": ("s_psp", "yolov5s_city_seg.yaml")}


def build(tag, yml, sd=None):
    from multiyolov5_b200.models.yolo import Model
    cfg = synth.load_cfg(yml)
    sd = sd or synth.synth_state_dict(synth.load_manifest(tag), cfg, seed=1)
    m = Model(yml)
    m.load_state_dict(sd)
    return m.cuda().eval(), cfg, sd


def rel(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


def fp32_truth(g, cfg, sd, x):
    """z and raw x_i of the fp32 reference, whole.  The fixture keeps every k-th row of them only (a max over a row sample would decide the
    comparison with the torch-fp16 yardstick by which anchors happen to be kept), so the whole arrays come from the fp32 CPU oracle, which
    must first reproduce every row the reference wrote (tolerances of test_oracle_golden's tensor-core-size test: raw stored as fp16)."""
    o = restate.model_forward(cfg, sd, x)
    truth = {"z": o["z"].numpy()} | {f"raw{i}": o["raw"][i].numpy() for i in range(3)}
    for k, tol in (("z", 2e-4), ("raw0", 1e-3), ("raw1", 1e-3), ("raw2", 1e-3)):
        assert rel(*fixture_pair(g, k, truth[k])) < tol, (k, rel(*fixture_pair(g, k, truth[k])))
    return truth


def errors_vs_fixture(z, raws, seg, g, truth):
    """every figure is against the fp32 reference (fixture, and `truth` for z / raw x_i).  raw / seg: max |err| / max |ref|; boxes: pixels;
    scores: absolute"""
    z = z.float().cpu().numpy(); zr = truth["z"]
    lo = torch.from_numpy(g["seg_lowres"])
    seg_ref = F.interpolate(lo, scale_factor=8, mode="bilinear", align_corners=True).numpy()      # models/yolo.py:163
    e = {f"raw{i}": rel(raws[i].float().cpu().numpy(), truth[f"raw{i}"]) for i in range(3)}
    e["seg"] = rel(seg.float().cpu().numpy(), seg_ref)
    # boxes in PIXELS.  The synthetic near-critical weights decode to boxes up to (2*sigmoid)^2 * anchor = 4 x 373 px wide, so the error is
    # reported (a) in pixels for object-sized boxes (<= 256 px) and (b) relative to the box size for all of them
    d = np.abs(z[..., :4] - zr[..., :4]).max(-1)
    size = np.maximum(zr[..., 2], zr[..., 3])
    small = size <= 256.0
    e["box_px_max_le256"] = float(d[small].max())
    e["box_px_p999"] = float(np.quantile(d, 0.999))
    e["box_rel_max"] = float((d / np.maximum(size, 8.0)).max())
    e["score_abs_max"] = float(np.abs(z[..., 4:] - zr[..., 4:]).max())
    e["cls_agree"] = float((seg.float().argmax(1).cpu().numpy() == g["seg_argmax"]).mean())
    return e


# measured on B200 x 1.5 (printed by the test; DESIGN.md section 4 keeps the table).  fp16 storage of ~60 layers of activations is what these
# are made of: the torch-fp16 yardstick below sits at the same level.
# measured (B200, profiles/parity_r2.md): raw <= 3.8e-3 (torch fp16: <= 5.2e-3), seg <= 2.6e-3 (3.4e-3), scores <= 1.43e-2 (2.2e-2), boxes <= 256 px:
# <= 2.4 px, class ids 99.38 % .. 100 % (99.55 % .. 99.998 %)
# boxes: worst of 32 256 anchors; a head-logit error of 0.05 moves w = (2 sigmoid)^2 * anchor by up to 7 % (ours <= 9.5 px on boxes <= 256 px and
# <= 7.0e-2 of the box size; torch fp16 <= 9.9 px and <= 9.9e-2)
CAPS = {"raw": 6e-3, "seg": 4e-3, "box_px_max_le256": 15.0, "box_rel_max": 0.11, "score_abs_max": 2.2e-2, "cls_agree_min": 0.99}


SCORE_CAP_E2E = 2.5e-2       # measured 1.2e-2 .. 1.4e-2 (sigmoid slope 1/4 x fp16-storage noise of the head logits)
EPS_SCORE, EPS_IOU = 2.5e-2, 4e-2   # what counts as 'within epsilon of a threshold' when the two detection sets are compared


@pytest.mark.parametrize("name", list(BIG))
def test_forward_vs_reference_fixture_at_tensor_core_sizes(name):
    tag, yml = BIG[name]
    g = np.load(os.path.join(synth.GOLDEN_DIR, f"netbig_{name}.npz"))
    B, H, W = [int(v) for v in g["shape"]]
    x = synth.synth_image(B, H, W, seed=int(g["seed"]))
    assert abs(float(x.double().sum()) - float(g["x_sum"])) < 1e-6 * float(g["x_sum"])
    model, cfg, sd = build(tag, yml)
    from multiyolov5_b200 import _lib
    (z, raws), seg = model(x.cuda())
    torch.cuda.synchronize()
    pb = model.engine().last_plan.pb
    n_conv = sum(1 for o in pb.ops if o.kind == _lib.OP_CONV)
    truth = fp32_truth(g, cfg, sd, x)
    ours = errors_vs_fixture(z, raws, seg, g, truth)
    # yardstick: the reference's own GPU configuration (fp16 weights / activations, torch + cuDNN kernels) on the same input
    sdc = {k: v.cuda() for k, v in sd.items()}
    y = restate.model_forward(cfg, sdc, x.cuda(), half=True)
    torch.cuda.synchronize()
    yard = errors_vs_fixture(y["z"], y["raw"], y["seg"], g, truth)
    print(f"\n[{name}] {n_conv} convs\n  ours  vs fp32 reference: {ours}\n  torch fp16 vs fp32 reference: {yard}")
    for k in ("raw0", "raw1", "raw2"):
        assert ours[k] <= CAPS["raw"], (k, ours[k])
        assert ours[k] <= 1.25 * yard[k] + 2e-4, (k, ours[k], yard[k])
    assert ours["seg"] <= CAPS["seg"] and ours["seg"] <= 1.25 * yard["seg"] + 2e-4, (ours["seg"], yard["seg"])
    for k in ("box_px_max_le256", "box_rel_max", "score_abs_max"):
        assert ours[k] <= CAPS[k], (k, ours[k])
        assert ours[k] <= 1.25 * yard[k] + 1e-3, (k, ours[k], yard[k])      # the reference's GPU path keeps `z` itself in fp16 (0.5 px steps above 512)
    assert ours["cls_agree"] >= CAPS["cls_agree_min"] and ours["cls_agree"] >= yard["cls_agree"] - 4e-3, (ours["cls_agree"], yard["cls_agree"])
    # taps: P5 features of the backbone / neck (fp16 fixtures)
    eng = model.engine()
    m2, _, _ = build(tag, yml, sd)
    m2.engine().noalias = True
    m2(x.cuda())
    for i in (9, 23):
        got = m2.engine().read_view(m2.engine().last_plan.pb.layer_views[i]).cpu().numpy()
        assert rel(*fixture_pair(g, f"layer{i}", got)) <= 8e-3, (i, rel(*fixture_pair(g, f"layer{i}", got)))


def _xyxy(z4):
    o = np.empty_like(z4)
    o[:, 0] = z4[:, 0] - z4[:, 2] / 2; o[:, 1] = z4[:, 1] - z4[:, 3] / 2
    o[:, 2] = z4[:, 0] + z4[:, 2] / 2; o[:, 3] = z4[:, 1] + z4[:, 3] / 2
    return o


def _iou(a, b):
    ix = np.maximum(0, np.minimum(a[2], b[:, 2]) - np.maximum(a[0], b[:, 0]))
    iy = np.maximum(0, np.minimum(a[3], b[:, 3]) - np.maximum(a[1], b[:, 1]))
    inter = ix * iy
    return inter / ((a[2] - a[0]) * (a[3] - a[1]) + (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1]) - inter + 1e-12)


def _explain_unmatched(d, z_other, dets_other, conf_thres, iou_thres, eps_c, eps_iou):
    """is detection `d` (x1,y1,x2,y2,conf,cls), absent from the other run's output, a threshold case there?  Looks the same anchor row up
    in the other run's predictions: its score within eps_c of conf_thres, or a kept box of the same class whose IoU with it is within eps_iou
    of iou_thres (suppressed there, kept here)."""
    boxes = _xyxy(z_other[:, :4])
    row = int(np.abs(boxes - d[None, :4]).sum(1).argmin())
    cls = int(d[5])
    conf_o = float(z_other[row, 4] * z_other[row, 5 + cls])
    if abs(conf_o - conf_thres) <= eps_c:
        return "score"
    best = z_other[row, 5:] * z_other[row, 4]
    if int(best.argmax()) != cls and abs(float(best.max()) - float(best[cls])) <= eps_c:
        return "class-tie"
    same = dets_other[dets_other[:, 5] == cls]
    if len(same) and np.any(np.abs(_iou(boxes[row], same[:, :4]) - iou_thres) <= eps_iou):
        return "iou"
    if len(dets_other) >= 300 and conf_o <= dets_other[:, 4].min() + eps_c:
        return "max_det"
    return None


def test_end_to_end_at_baseline_config_half_mode():
    """BASELINE.json configs[1]: yolov5s_city_seg (PSP), batch 16 x 3 x 512 x 1024, model.half() like detect.py:96-103, the bench's weights.
    Truth = the fp32 CPU oracle of the same 16 images + the reference's post-process."""
    import bench
    from multiyolov5_b200.models.yolo import Model
    from multiyolov5_b200.utils.general import non_max_suppression, seg_argmax
    yml, cfg, sd = bench.make_weights("s_psp")
    model = Model(yml)
    model.load_state_dict(sd)
    model.cuda().eval().half()
    B, H, W = 16, 512, 1024
    x = synth.synth_image(B, H, W, seed=21)
    (z, _), seg = model(x.cuda().half())
    dets = non_max_suppression(z, 0.25, 0.45)
    cls = seg_argmax(seg, (H, W))
    torch.cuda.synchronize()
    assert seg.dtype == torch.float16 and z.dtype == torch.float32
    torch.set_num_threads(min(32, os.cpu_count() or 1))
    zs, agree, lo_err = [], [], []
    n_unmatched = n_total = 0
    worst_px, sum_px, n_match, worst_score, worst_rel = 0.0, 0.0, 0, 0.0, 0.0
    reasons = {}
    for b in range(B):
        o = restate.model_forward(cfg, sd, x[b:b + 1])
        ref_cls = restate.seg_postprocess(o["seg"].numpy(), (H, W))[0]
        agree.append(float((cls[b].cpu().numpy() == ref_cls).mean()))
        zr = o["z"][0].numpy()
        zo = z[b].cpu().numpy()
        d_ref = restate.non_max_suppression(zr[None], 0.25, 0.45)[0]
        d_our = dets[b].cpu().numpy()
        n_total += len(d_ref)
        used = np.zeros(len(d_our), bool)
        for d in d_ref:                                     # every reference detection: same class, nearly the same box, among ours
            cand = np.where((d_our[:, 5] == d[5]) & ~used)[0]
            j = cand[np.abs(d_our[cand, :4] - d[None, :4]).max(1).argmin()] if len(cand) else -1
            size = max(float(d[2] - d[0]), float(d[3] - d[1]))
            if j >= 0 and np.abs(d_our[j, :4] - d[:4]).max() <= max(2.0, 0.03 * size):
                used[j] = True
                px = float(np.abs(d_our[j, :4] - d[:4]).max())
                if size <= 256.0:
                    worst_px = max(worst_px, px)
                worst_rel = max(worst_rel, px / max(size, 8.0))
                sum_px, n_match = sum_px + px, n_match + 1
                worst_score = max(worst_score, abs(float(d_our[j, 4]) - float(d[4])))
            else:
                why = _explain_unmatched(d, zo, d_our, 0.25, 0.45, EPS_SCORE, EPS_IOU)
                assert why is not None, f"image {b}: reference detection {d} missing from ours and not a threshold case"
                reasons[why] = reasons.get(why, 0) + 1
                n_unmatched += 1
        for j in np.where(~used)[0]:                        # and nothing extra that is not a threshold case in the reference run
            why = _explain_unmatched(d_our[j], zr, d_ref, 0.25, 0.45, EPS_SCORE, EPS_IOU)
            assert why is not None, f"image {b}: extra detection {d_our[j]} not explained by a threshold within epsilon"
            reasons[why] = reasons.get(why, 0) + 1
            n_unmatched += 1
    print(f"\n[e2e B=16 512x1024 half] class-id agreement min {min(agree):.5f} mean {np.mean(agree):.5f}; {n_total} reference detections, "
          f"{n_match} matched (box error max {worst_px:.3f} px on boxes <= 256 px, {worst_rel:.4f} of the box size overall, mean {sum_px / max(n_match, 1):.4f} px, score error max {worst_score:.4f}), "
          f"{n_unmatched} threshold cases {reasons}")
    assert min(agree) >= 0.982 and float(np.mean(agree)) >= 0.988, agree     # measured on B200: min 0.9881, mean 0.9920 (profiles/parity_r2.md)
    assert n_total > 200 and n_unmatched <= 0.03 * n_total + 2
    assert worst_px <= 3.7 and worst_rel <= 4.2e-2 and worst_score <= SCORE_CAP_E2E      # measured 2.44 px / 2.8e-2 / 1.7e-2 (x 1.5)
