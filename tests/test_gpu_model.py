"""GPU: Model(cfg).forward on the compiled sm_100a plan vs (a) the fp16-storage emulation of the oracle (tight: only fp32
accumulation order differs) and (b) the fixtures produced by the unmodified fp32 reference (north_star budget; measured
deviations are recorded in DESIGN.md)."""
import os

import numpy as np
import pytest
import torch

from oracle import restate, synth
from oracle.digest import fixture_pair, fixture_shape

pytestmark = pytest.mark.gpu
NETS = {"s_psp": "yolov5s_city_seg.yaml", "m_lab": "yolov5m_city_seg_lab.yaml", "s_bise": "yolov5s_city_seg_bise.yaml",
        "s_base": "yolov5s_city_seg_base.yaml", "m_psp": "yolov5m_city_seg.yaml"}


def relmax(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


def build(tag):
    from multiyolov5_b200.models.yolo import Model
    cfg = synth.load_cfg(NETS[tag])
    sd = synth.synth_state_dict(synth.load_manifest(tag), cfg, seed=1)
    m = Model(NETS[tag])
    m.load_state_dict(sd)
    return m.cuda().eval(), cfg, sd


def layerwise_report(model, cfg, sd, x, upto=24):
    """first top-level layer whose output deviates from the fp16-emulation oracle (debug aid for failures)."""
    o = restate.model_forward(cfg, sd, x.cpu(), quantised=True, keep=tuple(range(upto)))
    from multiyolov5_b200.models.yolo import Model
    model = Model(model.yaml).cuda().eval()
    model.load_state_dict(sd)
    eng = model.engine()
    eng.noalias = True
    model(x)
    lines = []
    for i in range(upto):
        v = eng.last_plan.pb.layer_views[i]
        if v is None:
            continue
        got = eng.read_view(v).cpu().numpy()
        lines.append(f"L{i}: rel {relmax(got, o['layers'][i].numpy()):.2e}")
    return " | ".join(lines)


@pytest.mark.parametrize("tag", list(NETS))
def test_forward_matches_reference_fixture(tag):
    model, cfg, sd = build(tag)
    g = np.load(os.path.join(synth.GOLDEN_DIR, f"net_{tag}.npz"))
    x = torch.from_numpy(g["x"]).cuda()
    (z, raw), seg = model(x)
    torch.cuda.synchronize()
    q = restate.model_forward(cfg, sd, x.cpu(), quantised=True)
    # (a) vs fp16-emulation oracle: kernels are right iff this is tight
    ea = dict(seg=relmax(seg.cpu().numpy(), q["seg"].numpy()), z=relmax(z.cpu().numpy(), q["z"].numpy()),
              raw0=relmax(raw[0].cpu().numpy(), q["raw"][0].numpy()))
    # (b) vs the unmodified fp32 reference (fixture)
    eb = dict(seg=relmax(*fixture_pair(g, "seg", seg.cpu().numpy())), z=relmax(z.cpu().numpy(), g["z"]), raw0=relmax(raw[0].cpu().numpy(), g["raw0"]))
    print(f"\n[{tag}] vs fp16-emulation oracle {ea}  vs fp32 reference {eb}")
    if max(ea.values()) > 4e-3:
        print(layerwise_report(model, cfg, sd, x))
    assert raw[0].shape == g["raw0"].shape and raw[2].shape == g["raw2"].shape and seg.shape == fixture_shape(g, "seg")
    assert max(ea.values()) <= 4e-3, ea
    assert max(eb.values()) <= 2e-2, eb


@pytest.mark.parametrize("tag,hw", [("s_psp", (256, 512)), ("m_lab", (256, 256))])
def test_forward_tensor_core_sizes(tag, hw):
    """resolution where every backbone/neck/head conv takes the tcgen05 path (P5 = 8x16 >= one 128-pixel tile)."""
    model, cfg, sd = build(tag)
    x = synth.synth_image(2, hw[0], hw[1], seed=3).cuda()
    (z, raw), seg = model(x)
    torch.cuda.synchronize()
    q = restate.model_forward(cfg, sd, x.cpu(), quantised=True)
    f = restate.model_forward(cfg, sd, x.cpu(), quantised=False)
    ea = dict(seg=relmax(seg.cpu().numpy(), q["seg"].numpy()), z=relmax(z.cpu().numpy(), q["z"].numpy()),
              raw2=relmax(raw[2].cpu().numpy(), q["raw"][2].numpy()))
    eb = dict(seg=relmax(seg.cpu().numpy(), f["seg"].numpy()), z=relmax(z.cpu().numpy(), f["z"].numpy()))
    print(f"\n[{tag} {hw}] vs fp16-emulation oracle {ea}  vs fp32 oracle {eb}")
    if max(ea.values()) > 4e-3:
        print(layerwise_report(model, cfg, sd, x))
    assert max(ea['seg'], ea['raw2']) <= 4e-3 and ea['z'] <= 2e-2, ea   # z amplifies raw-logit noise through (2*sigmoid)^2*anchor
    assert max(eb.values()) <= 2e-2, eb
    # fused argmax == argmax of the materialised logits (bit-exact class ids)
    out = model(x, seg_argmax=True)
    assert torch.equal(out[2], seg.argmax(1))


@pytest.mark.parametrize("tag", list(NETS))
def test_forward_full_resolution_all_heads(tag):
    """BASELINE.json resolution (512x1024): every head / model size on the tensor-core path incl. strip mode, vertical rounds,
    dilation 6/9 (Lab ASPP), the BiSe global branch and C3SPP (Base)."""
    model, cfg, sd = build(tag)
    x = synth.synth_image(1, 512, 1024, seed=7).cuda()
    (z, raw), seg = model(x)
    torch.cuda.synchronize()
    q = restate.model_forward(cfg, sd, x.cpu(), quantised=True)
    ea = dict(seg=relmax(seg.cpu().numpy(), q["seg"].numpy()), raw0=relmax(raw[0].cpu().numpy(), q["raw"][0].numpy()),
              raw2=relmax(raw[2].cpu().numpy(), q["raw"][2].numpy()), z=relmax(z.cpu().numpy(), q["z"].numpy()))
    print(f"\n[{tag} 512x1024] vs fp16-emulation oracle {ea}")
    assert z.shape == (1, 32256, 15) and seg.shape == (1, 19, 512, 1024)
    assert max(ea["seg"], ea["raw0"], ea["raw2"]) <= 6e-3 and ea["z"] <= 3e-2, ea
    # second call replays the captured CUDA graph: must reproduce the eager first call bit for bit
    (z2, raw2), seg2 = model(x)
    assert torch.equal(z, z2) and torch.equal(seg, seg2)


@pytest.mark.parametrize("tag,dtype", [("s_psp", torch.float32), ("s_psp", torch.uint8), ("m_psp", torch.float16)])
def test_fused_layer0_matches_unfused_path(tag, dtype, monkeypatch):
    """csrc/focus_conv.cu (Focus + conv in one kernel from the NCHW image) vs the space-to-depth kernel + tcgen05 conv."""
    model, cfg, sd = build(tag)
    x8 = torch.randint(0, 256, (2, 3, 128, 256), dtype=torch.uint8, generator=torch.Generator().manual_seed(3)).cuda()
    x = x8 if dtype == torch.uint8 else (x8.float() / 255.0).to(dtype)
    monkeypatch.setenv("MYOLO_FOCUS_FUSION", "1")
    eng = model.engine()
    eng.noalias = True          # keep layer 0's buffer readable after the forward
    model(x)
    y_fused = eng.read_view(eng.last_plan.pb.layer_views[0]).clone()
    monkeypatch.setenv("MYOLO_FOCUS_FUSION", "0")
    model2, _, _ = build(tag)
    model2.engine().noalias = True
    model2(x)
    y_ref = model2.engine().read_view(model2.engine().last_plan.pb.layer_views[0])
    from multiyolov5_b200 import _lib
    assert any(o.kind == _lib.OP_FOCUS_CONV for o in eng.last_plan.pb.ops) and not any(o.kind == _lib.OP_FOCUS_CONV for o in model2.engine().last_plan.pb.ops)
    o = restate.model_forward(cfg, sd, (x8.float() / 255.0).cpu(), quantised=True, keep=(0,))["layers"][0].numpy()
    assert relmax(y_fused.cpu().numpy(), o) < 3e-3 and relmax(y_ref.cpu().numpy(), o) < 3e-3


def test_half_mode_like_reference_cuda_path():
    """detect.py:96-103: model.half() + img.half() -> fp16 seg logits; class ids must agree with the fp32-IO run except at near-ties."""
    model, cfg, sd = build("s_psp")
    x = synth.synth_image(2, 256, 512, seed=9).cuda()
    (z32, _), seg32 = model(x)
    mh, _, _ = build("s_psp")
    mh.half()
    (z16, _), seg16 = mh(x.half())
    torch.cuda.synchronize()
    assert seg16.dtype == torch.float16 and seg32.dtype == torch.float32
    assert relmax(seg16.float().cpu().numpy(), seg32.cpu().numpy()) < 4e-3
    assert relmax(z16.cpu().numpy(), z32.cpu().numpy()) < 2e-2
    from multiyolov5_b200.utils.general import seg_argmax
    a16, a32 = seg_argmax(seg16), seg_argmax(seg32)
    assert torch.equal(a16, seg16.float().argmax(1))            # fp16 fast path is an exact argmax of what it is given
    assert (a16 != a32).float().mean().item() < 1e-2   # near-tie pixels flip under fp16 rounding of the logits (0.35% measured)


def test_simt_and_tensor_core_paths_agree(monkeypatch):
    model, cfg, sd = build("s_psp")
    x = synth.synth_image(1, 256, 512, seed=4).cuda()
    (z, raw), seg = model(x)
    monkeypatch.setenv("MYOLO_FORCE_SIMT", "1")
    model2, _, _ = build("s_psp")
    (z2, raw2), seg2 = model2(x)
    torch.cuda.synchronize()
    assert relmax(seg.cpu().numpy(), seg2.cpu().numpy()) < 4e-3
    assert relmax(z.cpu().numpy(), z2.cpu().numpy()) < 2e-2
    assert relmax(raw[0].cpu().numpy(), raw2[0].cpu().numpy()) < 4e-3


@pytest.mark.parametrize("tag", ["s_psp", "m_lab"])
def test_c3_cv1_cv2_fusion_matches_separate_launches(tag, monkeypatch):
    """planner option MYOLO_FUSE_C3: the two 1x1 convs of a C3 that read the same input run as ONE conv with concatenated output channels
    (reference models/common.py:138-139 computes them separately).  Same K loop per output channel -> same values."""
    hw = (256, 512)
    monkeypatch.setenv("MYOLO_FUSE_C3", "0")
    model, cfg, sd = build(tag)
    x = synth.synth_image(2, hw[0], hw[1], seed=11).cuda()
    (z, raw), seg = model(x)
    n0 = len(model.engine().last_plan.pb.ops)
    monkeypatch.setenv("MYOLO_FUSE_C3", "1")
    model2, _, _ = build(tag)
    (z2, raw2), seg2 = model2(x)
    torch.cuda.synchronize()
    n1 = len(model2.engine().last_plan.pb.ops)
    assert n1 < n0, (n0, n1)
    assert relmax(seg2.cpu().numpy(), seg.cpu().numpy()) < 1e-5 and relmax(z2.cpu().numpy(), z.cpu().numpy()) < 1e-5
    assert relmax(raw2[2].cpu().numpy(), raw[2].cpu().numpy()) < 1e-5


def test_no_cpu_path():
    from multiyolov5_b200 import _lib
    model, _, _ = build("s_psp")
    with pytest.raises(_lib.MyoloError):
        model(torch.zeros(1, 3, 64, 64))
