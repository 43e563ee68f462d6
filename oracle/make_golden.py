"""TEST INFRASTRUCTURE — generates tests/golden/* by running the UNMODIFIED reference (imported from
/root/reference through oracle/ref_shims.py) in the build container.  The reference ships no golden
vectors (SURVEY.md §4), so these fixtures are what pins the oracle restatement and the CUDA path.

    python oracle/make_golden.py            # regenerate everything (needs /root/reference)

Fixtures (all small; weights are NOT stored — they are re-synthesised from the manifest + seed):
  manifest_<tag>.json      reference state_dict keys / shapes / dtypes for each model config
  net_<tag>.npz            input, z, raw x_i, seg (+ low-res logits, a few layer outputs) of Model.forward (eval, fused)
  nms_cases.npz            non_max_suppression inputs/outputs for several flag combinations
  segpost_cases.npz        detect.py:191-193 upsample+argmax inputs/outputs
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import ref_shims, synth  # noqa: E402

GOLD = os.path.join(HERE, "..", "tests", "golden")

# tag -> (yaml in multiyolov5_b200/models, reference yaml, head line to enable, B, H, W)
NET_CASES = {
    "s_psp": ("yolov5s_city_seg.yaml", "SegMaskPSP", 2, 64, 96),
    "m_lab": ("yolov5m_city_seg_lab.yaml", "SegMaskLab", 1, 64, 64),
    "s_bise": ("yolov5s_city_seg_bise.yaml", "SegMaskBiSe", 1, 64, 64),
    "s_base": ("yolov5s_city_seg_base.yaml", "SegMaskBase", 1, 64, 64),
    "m_psp": ("yolov5m_city_seg.yaml", "SegMaskPSP", 1, 64, 64),
}
KEEP_LAYERS = (0, 4, 9, 17, 23)


def build_reference_model(ref_yolo, cfg: dict):
    import copy
    return ref_yolo.Model(copy.deepcopy(cfg))


def gen_nets(ref_yolo):
    for tag, (yml, head, B, H, W) in NET_CASES.items():
        cfg = synth.load_cfg(yml)
        torch.manual_seed(0)
        model = build_reference_model(ref_yolo, cfg)
        sd0 = model.state_dict()
        manifest = [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in sd0.items()]
        with open(os.path.join(GOLD, f"manifest_{tag}.json"), "w") as f:
            json.dump(manifest, f)
        sd = synth.synth_state_dict(manifest, cfg, seed=1)
        # anchors buffers must equal what the reference itself computed
        for k in sd:
            if k.endswith(".anchors") or k.endswith(".anchor_grid"):
                assert torch.allclose(sd[k], sd0[k]), k
        model.load_state_dict(sd)
        model.fuse().eval()
        x = synth.synth_image(B, H, W, seed=0)
        feats = {}
        hooks = [model.model[i].register_forward_hook(lambda m, a, o, i=i: feats.__setitem__(i, o.detach().clone()))
                 for i in KEEP_LAYERS]
        lowres = {}
        seg_head = model.model[24]
        seq = seg_head.out if hasattr(seg_head, "out") else (seg_head.decoder if hasattr(seg_head, "decoder") else seg_head.m)
        hooks.append(seq[-1].register_forward_hook(lambda m, a, o: lowres.__setitem__("x", a[0].detach().clone())))
        with torch.no_grad():
            out = model(x)
        for h in hooks:
            h.remove()
        (z, raw), seg = out
        arrs = dict(x=x.numpy(), z=z.numpy(), seg=seg.numpy(), seg_lowres=lowres["x"].numpy())
        for i, r in enumerate(raw):
            arrs[f"raw{i}"] = r.numpy()
        for i, t in feats.items():
            arrs[f"layer{i}"] = t.numpy().astype(np.float16)  # layer taps stored as fp16 to keep fixtures small
        if arrs["seg"].nbytes > 512 * 1024:
            keep_rows(arrs, "seg", 3)
        np.savez_compressed(os.path.join(GOLD, f"net_{tag}.npz"), **arrs)
        print(tag, "params", sum(v.numel() for v in sd0.values()), {k: v.shape for k, v in arrs.items()},
              "z|max|", float(z.abs().max()), "seg std", float(seg.std()))


def gen_nms(ref_general):
    cases = {}
    pred = synth.synth_predictions(2, 3000, seed=0)
    pred[1, ::7, 4] = 0.1  # some rows below conf
    pred[0, 100:110] = pred[0, 90:100]  # exact duplicates -> score ties, stable order matters
    settings = {
        "default": dict(conf_thres=0.25, iou_thres=0.45),
        "test_ml": dict(conf_thres=0.001, iou_thres=0.6, multi_label=True),
        "agnostic": dict(conf_thres=0.4, iou_thres=0.5, agnostic=True),
        "classes": dict(conf_thres=0.25, iou_thres=0.45, classes=[0, 3, 7]),
        "none_pass": dict(conf_thres=1.5, iou_thres=0.45),
    }
    small = synth.synth_predictions(2, 400, seed=3)
    cases["pred_big"] = pred
    cases["pred_small"] = small
    for name, kw in settings.items():
        for pn, p in (("big", pred), ("small", small)):
            if name == "test_ml" and pn == "big":
                continue  # 30k candidates x greedy numpy oracle is slow; the small case covers the flag
            outs = ref_general.non_max_suppression(torch.from_numpy(p.copy()), **kw)
            for b, o in enumerate(outs):
                cases[f"out_{name}_{pn}_{b}"] = o.numpy()
            print("nms", name, pn, [tuple(o.shape) for o in outs])
    with open(os.path.join(GOLD, "nms_settings.json"), "w") as f:
        json.dump(settings, f)
    np.savez_compressed(os.path.join(GOLD, "nms_cases.npz"), **cases)


def gen_segpost():
    import torch.nn.functional as F
    rs = np.random.RandomState(5)
    cases = {}
    for name, (c, h, w, H, W) in {"x8": (19, 16, 32, 128, 256), "odd": (19, 9, 13, 40, 77), "same": (19, 24, 24, 24, 24),
                                  "up2": (19, 32, 64, 64, 128)}.items():
        seg = rs.normal(0, 2, (1, c, h, w)).astype(np.float32)
        up = F.interpolate(torch.from_numpy(seg), (H, W), mode="bilinear", align_corners=True)[0]
        am = up.max(axis=0)[1]
        cases[f"in_{name}"] = seg
        if name in ("odd", "same"):
            cases[f"up_{name}"] = up.numpy()
        cases[f"argmax_{name}"] = am.numpy().astype(np.uint8)
    np.savez_compressed(os.path.join(GOLD, "segpost_cases.npz"), **cases)
    print("segpost", list(cases))


def load_reference_loss():
    """utils/loss.py of the reference, executed from where it lies with ONE in-memory textual fix: `gj.clamp_(0, gain[3] - 1)`
    (utils/loss.py:212) passes a float tensor as the bound of a long tensor, which torch >= 1.12 rejects; `int(gain[k]) - 1` has the
    same value (SURVEY.md section 8c).  Nothing is written to disk."""
    import types
    src = open(os.path.join(ref_shims.REF_ROOT, "utils", "loss.py")).read()
    assert "gain[3] - 1" in src and "gain[2] - 1" in src
    src = src.replace("gain[3] - 1", "int(gain[3]) - 1").replace("gain[2] - 1", "int(gain[2]) - 1")
    mod = types.ModuleType("ref_loss_patched")
    exec(compile(src, "reference:utils/loss.py", "exec"), mod.__dict__)
    return mod


def loss_hyp(nl=3, nc=10, imgsz=1024):
    """data/hyp.scratch.yaml with the scalings of train.py:248-251 (imgsz = the long side, train.py:196)"""
    import yaml
    with open(os.path.join(ref_shims.REF_ROOT, "data", "hyp.scratch.yaml")) as f:
        hyp = yaml.safe_load(f)
    hyp["box"] *= 3.0 / nl
    hyp["cls"] *= nc / 80.0 * 3.0 / nl
    hyp["obj"] *= (imgsz / 640) ** 2 * 3.0 / nl
    hyp["label_smoothing"] = 0.0
    return hyp


def gen_loss(ref_yolo):
    """ComputeLoss.__call__ (utils/loss.py:115-162) + SegmentationLosses.forward (:235-237) on small seeded inputs; stores the loss,
    loss_items and d(loss)/d(prediction) so both the restatement and the product loss can be checked."""
    ref_loss = load_reference_loss()
    cfg = synth.load_cfg("yolov5s_city_seg.yaml")
    torch.manual_seed(0)
    model = build_reference_model(ref_yolo, cfg)
    hyp = loss_hyp(nl=3, nc=cfg["nc"], imgsz=256)
    model.hyp, model.gr, model.nc = hyp, 1.0, cfg["nc"]
    det = model.model[-1]
    crit = ref_loss.ComputeLoss(model)
    rs = np.random.RandomState(3)
    B, H, W = 2, 128, 256
    cases = {"hyp_json": np.frombuffer(json.dumps(hyp).encode(), dtype=np.uint8), "anchors": det.anchors.numpy().copy(),
             "strides": det.stride.numpy().copy()}
    for name, nt in (("a", 24), ("empty", 0), ("edge", 16)):
        p = [torch.from_numpy(rs.normal(0, 1.0, (B, det.na, H // s, W // s, det.no)).astype(np.float32)).requires_grad_(True)
             for s in (8, 16, 32)]
        t = np.zeros((nt, 6), np.float32)
        if nt:
            t[:, 0] = rs.randint(0, B, nt)
            t[:, 1] = rs.randint(0, cfg["nc"], nt)
            t[:, 2:4] = rs.uniform(0.02, 0.98, (nt, 2)) if name != "edge" else rs.choice([0.001, 0.5, 0.999, 0.26, 0.74], (nt, 2))
            t[:, 4:6] = rs.uniform(0.02, 0.5, (nt, 2))
        loss, items = crit(p, torch.from_numpy(t))
        loss.backward()
        cases[f"{name}_targets"] = t
        for i in range(3):
            cases[f"{name}_p{i}"] = p[i].detach().numpy()
            cases[f"{name}_g{i}"] = p[i].grad.numpy()
        cases[f"{name}_loss"] = loss.detach().numpy()
        cases[f"{name}_items"] = items.numpy()
    # segmentation CE (ignore_index=-1)
    seg = torch.from_numpy(rs.normal(0, 2.0, (2, 19, 32, 64)).astype(np.float32)).requires_grad_(True)
    mask = torch.from_numpy(rs.randint(-1, 19, (2, 32, 64)).astype(np.int64))
    sl = ref_loss.SegmentationLosses(ignore_index=-1)(seg, mask)
    sl.backward()
    np.savez_compressed(os.path.join(GOLD, "loss_cases.npz"), **cases)
    np.savez_compressed(os.path.join(GOLD, "seg_loss_cases.npz"), seg_logits=seg.detach().numpy(), seg_mask=mask.numpy(),
                        seg_loss=sl.detach().numpy(), seg_grad=seg.grad.numpy())      # a file of its own: each stays under 1 MB
    print("loss", {k: v.shape for k, v in cases.items() if "loss" in k or "items" in k}, "seg", float(sl))


def gen_letterbox():
    """the reference's own `letterbox` (utils/datasets.py:818-848, cv2 underneath) on small synthetic frames + one photo crop"""
    import cv2
    import utils.datasets as ref_datasets     # the reference's module (sys.path set by import_reference)
    rs = np.random.RandomState(9)
    cases = {}
    photo = cv2.imread(os.path.join(ref_shims.REF_ROOT, "data", "images", "bus.jpg"))
    frames = {"rand_a": rs.randint(0, 256, (97, 131, 3), dtype=np.uint8), "rand_b": rs.randint(0, 256, (128, 256, 3), dtype=np.uint8),
              "photo": np.ascontiguousarray(photo[200:360, 300:520]) if photo is not None else rs.randint(0, 256, (160, 220, 3), dtype=np.uint8),
              "smooth": (np.add.outer(np.arange(150), np.arange(90))[..., None] * np.array([1, 2, 3]) % 256).astype(np.uint8)}
    settings = {"a64": dict(new_shape=64, stride=32), "half": dict(new_shape=(64, 128), stride=32), "up": dict(new_shape=192, stride=32),
                "noauto": dict(new_shape=(96, 160), auto=False), "fill": dict(new_shape=(80, 112), auto=False, scaleFill=True),
                "noup": dict(new_shape=320, scaleup=False, stride=64)}
    meta = {}
    for fn, frame in frames.items():
        cases[f"in_{fn}"] = frame
        for sn, kw in settings.items():
            out, ratio, dwdh = ref_datasets.letterbox(frame.copy(), **kw)
            cases[f"out_{fn}_{sn}"] = out
            meta[f"{fn}_{sn}"] = dict(kw=kw, ratio=[float(ratio[0]), float(ratio[1])], dwdh=[float(dwdh[0]), float(dwdh[1])])
    cases["meta_json"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(GOLD, "letterbox_cases.npz"), **cases)
    print("letterbox", len(meta), "cases")


def gen_consumers():
    """seg output consumers (SURVEY.md section 8f rank 2): the reference's label2image / trainid2id (detect.py:69-77), the blend
    cv2.addWeighted(mask, 0.4, im0, 0.6, 0) (detect.py:194) and batch_pix_accuracy / batch_intersection_union (utils/metrics.py:234-275)"""
    import importlib
    import cv2
    det = importlib.import_module("detect")
    met = importlib.import_module("utils.metrics")
    rs = np.random.RandomState(21)
    cases = {"colormap": np.array(det.Cityscapes_COLORMAP, np.uint8), "idmap": np.array(det.Cityscapes_IDMAP, np.uint8)}
    pred = rs.randint(0, 19, (96, 160)).astype(np.int64)
    im0 = rs.randint(0, 256, (96, 160, 3), dtype=np.uint8)
    mask = det.label2image(pred, det.Cityscapes_COLORMAP)[:, :, ::-1]
    cases.update(pred=pred, im0=im0, mask_bgr=np.ascontiguousarray(mask), ids=det.trainid2id(pred, det.Cityscapes_IDMAP),
                 blend=cv2.addWeighted(np.ascontiguousarray(mask), 0.4, im0, 0.6, 0))
    out = torch.from_numpy(rs.normal(0, 1, (2, 19, 48, 64)).astype(np.float32))
    tgt = torch.from_numpy(rs.randint(-1, 19, (2, 48, 64)).astype(np.int64))
    correct, labeled = met.batch_pix_accuracy(out, tgt)
    inter, union = met.batch_intersection_union(out, tgt, 19)
    cases.update(m_out=out.numpy(), m_tgt=tgt.numpy(), m_correct=np.int64(correct), m_labeled=np.int64(labeled), m_inter=inter.astype(np.int64),
                 m_union=union.astype(np.int64))
    np.savez_compressed(os.path.join(GOLD, "consumer_cases.npz"), **cases)
    print("consumers", int(correct), int(labeled), inter[:4], union[:4])


# tcgen05-sized inference fixtures: every backbone / neck / head conv of these inputs runs on conv_tc_kernel (the 64x96 fixtures above
# put every map below P2 on the CUDA-core kernel).  Stored compactly: z fp32, raw x_i fp16, low-resolution seg logits fp32, two taps;
# z, raw x_i and the taps keep every `step`-th row (keep_rows) so that each fixture stays under 1 MB.
BIG_CASES = {     # name: (tag, yaml, B, H, W, input seed, row step)
    "s_psp_256x512": ("s_psp", "yolov5s_city_seg.yaml", 1, 256, 512, 3, 3),
    "m_lab_256x512": ("m_lab", "yolov5m_city_seg_lab.yaml", 1, 256, 512, 3, 3),
    "s_psp_512x1024": ("s_psp", "yolov5s_city_seg.yaml", 1, 512, 1024, 7, 13),
}


def gen_nets_big(ref_yolo):
    for name, (tag, yml, B, H, W, seed, step) in BIG_CASES.items():
        cfg = synth.load_cfg(yml)
        torch.manual_seed(0)
        model = build_reference_model(ref_yolo, cfg)
        sd = synth.synth_state_dict(synth.load_manifest(tag), cfg, seed=1)
        model.load_state_dict(sd)
        model.fuse().eval()
        x = synth.synth_image(B, H, W, seed=seed)       # NOT stored: re-created from the seed by the tests (checksum below)
        feats, lowres = {}, {}
        hooks = [model.model[i].register_forward_hook(lambda m, a, o, i=i: feats.__setitem__(i, o.detach().clone())) for i in (9, 23)]
        seg_head = model.model[24]
        seq = seg_head.out if hasattr(seg_head, "out") else (seg_head.decoder if hasattr(seg_head, "decoder") else seg_head.m)
        hooks.append(seq[-1].register_forward_hook(lambda m, a, o: lowres.__setitem__("x", a[0].detach().clone())))
        with torch.no_grad():
            (z, raw), seg = model(x)
        for h in hooks:
            h.remove()
        arrs = dict(x_sum=np.float64(x.double().sum().item()), z=z.numpy(), seg_lowres=lowres["x"].numpy(),
                    seg_argmax=seg.argmax(1).numpy().astype(np.uint8), seed=np.int64(seed), shape=np.array([B, H, W]))
        for i, r in enumerate(raw):
            arrs[f"raw{i}"] = r.numpy().astype(np.float16)
            arrs[f"raw{i}_absmax"] = np.float32(r.abs().max().item())
        for i, t in feats.items():
            arrs[f"layer{i}"] = t.numpy().astype(np.float16)
        for k in ("z", "raw0", "raw1", "raw2", "layer9", "layer23"):
            keep_rows(arrs, k, step)
        np.savez_compressed(os.path.join(GOLD, f"netbig_{name}.npz"), **arrs)
        print(name, {k: getattr(v, "shape", None) for k, v in arrs.items()}, os.path.getsize(os.path.join(GOLD, f"netbig_{name}.npz")) / 1e6, "MB")


TRAIN_CASES = {"s_psp": "yolov5s_city_seg.yaml", "s_bise": "yolov5s_city_seg_bise.yaml", "m_lab": "yolov5m_city_seg_lab.yaml",
               "s_base": "yolov5s_city_seg_base.yaml"}


from oracle.digest import grad_digest, keep_rows, train_probe_tensors  # noqa: E402


def gen_train(ref_yolo):
    """the reference's own TRAIN-mode `Model` (batch-statistics BatchNorm, active Dropout) + torch.autograd on a small input: head outputs,
    the gradient of every parameter (digest), and the BatchNorm running statistics after the forward.  Pins
    oracle.restate.model_forward_train (tests/test_oracle_golden.py)."""
    for tag, yml in TRAIN_CASES.items():
        cfg = synth.load_cfg(yml)
        torch.manual_seed(0)
        model = build_reference_model(ref_yolo, cfg)
        sd = synth.synth_state_dict(synth.load_manifest(tag), cfg, seed=1, gain=1.0)
        model.load_state_dict(sd)
        model.train()
        x = synth.synth_image(2, 64, 96, seed=5)
        masks, pre = [], []
        hooks = []
        for m in model.modules():
            if isinstance(m, torch.nn.Dropout):    # the Base head's Dropout is in place (models/yolo.py:140): keep a copy of its input
                hooks.append(m.register_forward_pre_hook(lambda mod, a: pre.append(a[0].detach().clone())))
                hooks.append(m.register_forward_hook(lambda mod, a, o: masks.append(((o != 0) | (pre[-1] == 0)).detach().clone())))
        torch.manual_seed(123)
        out = model(x)
        for h in hooks:
            h.remove()
        raws, seg = out
        segs = list(seg) if isinstance(seg, (list, tuple)) else [seg]
        Rs, Ss = train_probe_tensors([tuple(r.shape) for r in raws], [tuple(g.shape) for g in segs])
        loss = sum((r * R).sum() for r, R in zip(raws, Rs)) + sum((g * S).sum() for g, S in zip(segs, Ss))
        loss.backward()
        arrs = {"loss": np.float64(loss.item())}
        for i, r in enumerate(raws):
            arrs[f"raw{i}"] = r.detach().numpy()
        for k, g in enumerate(segs):
            arrs[f"seg{k}_sub"] = g.detach()[:, :, ::3, ::3].numpy()
        names, digests = [], []
        for n, p_ in model.named_parameters():
            if p_.grad is not None:
                names.append(n)
                digests.append(grad_digest(p_.grad))
        arrs["grad_names"] = np.array(names)
        arrs["grad_digest"] = np.stack(digests)
        rn, rm, rv = [], [], []
        for n, m in model.named_modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                rn.append(n)
                rm.append(m.running_mean.numpy().copy())
                rv.append(m.running_var.numpy().copy())
        arrs["bn_names"] = np.array(rn)
        arrs["bn_mean"] = np.concatenate(rm)
        arrs["bn_var"] = np.concatenate(rv)
        if masks:
            assert len(masks) == 1
            arrs["dropout_keep_bits"] = np.packbits(masks[0].numpy().astype(np.uint8).reshape(-1))
            arrs["dropout_shape"] = np.array(masks[0].shape)
        np.savez_compressed(os.path.join(GOLD, f"train_{tag}.npz"), **arrs)
        print("train", tag, "loss", float(loss), len(names), "grads", len(rn), "BN layers", os.path.getsize(os.path.join(GOLD, f"train_{tag}.npz")) / 1e6, "MB")


def gen_ckpt(ref_yolo):
    """a checkpoint exactly as the reference's train.py:482-494 writes it (whole pickled reference `Model` in half precision inside a
    dict), for a quarter-width yolov5s_city_seg whose backbone / neck stop at 128 yaml channels (32 after the width multiple; every conv
    keeps >= 16 channels) so the fixture stays under 1 MB, plus what the reference's own `attempt_load` recipe
    (`ckpt['model'].float().fuse().eval()`, models/experimental.py:119) computes from it on a small input."""
    import copy
    cfg = synth.load_cfg("yolov5s_city_seg.yaml")
    cfg["width_multiple"] = 0.25
    for row in cfg["backbone"] + cfg["head"]:
        if row[2] in ("Focus", "Conv", "C3", "SPP"):
            row[3][0] = min(row[3][0], 128)
    torch.manual_seed(7)
    model = build_reference_model(ref_yolo, cfg)
    g = torch.Generator().manual_seed(11)
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.1)
                m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) + 0.5)
                m.weight.copy_(torch.rand(m.weight.shape, generator=g) * 0.4 + 0.8)
                m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
            elif isinstance(m, torch.nn.Conv2d):
                fan_in = m.weight.shape[1] * m.weight.shape[2] * m.weight.shape[3]
                m.weight.copy_(torch.randn(m.weight.shape, generator=g) * (2.0 / fan_in) ** 0.5)
    model.names = [f"cls{i}" for i in range(cfg["nc"])]
    ckpt = {"epoch": 3, "best_fitness": 0.5, "training_results": "synthetic", "model": copy.deepcopy(model).half(), "ema": None, "updates": 0,
            "optimizer": None, "wandb_id": None}
    path = os.path.join(GOLD, "ref_ckpt_tiny.pt")
    torch.save(ckpt, path)
    m2 = torch.load(path, weights_only=False)["model"].float().fuse().eval()     # the reference's own loading recipe
    x = synth.synth_image(1, 64, 64, seed=5)
    with torch.no_grad():
        (z, raw), seg = m2(x)
    np.savez_compressed(os.path.join(GOLD, "ref_ckpt_tiny_out.npz"), z=z.numpy(), seg=seg.numpy(), raw0=raw[0].numpy(),
                        names=np.array(model.names), stride=model.stride.numpy())
    print("ckpt", os.path.getsize(path) / 1e6, "MB", z.shape, seg.shape)


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    cwd = os.getcwd()
    ref_yolo, ref_general = ref_shims.import_reference()
    only = set(sys.argv[1:])
    if not only or "nets" in only:
        gen_nets(ref_yolo)
    if not only or "nms" in only:
        gen_nms(ref_general)
    if not only or "segpost" in only:
        gen_segpost()
    if not only or "loss" in only:
        gen_loss(ref_yolo)
    if not only or "letterbox" in only:
        gen_letterbox()
    if not only or "consumers" in only:
        gen_consumers()
    if not only or "ckpt" in only:
        gen_ckpt(ref_yolo)
    if not only or "netsbig" in only:
        gen_nets_big(ref_yolo)
    if not only or "train" in only:
        gen_train(ref_yolo)
