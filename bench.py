#!/usr/bin/env python
"""Benchmark of the hot path: images/sec @1024x512 (det+seg forward + NMS + seg argmax == reference detect.py:144-148,191-193).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--cfg s_psp|m_lab] [--batch B] [--dump-outputs DIR]

N=1 workload = BASELINE.json configs[1]: yolov5s_city_seg.yaml (PSP head), batch 16 x 3 x 512 x 1024 synthetic, fp16 storage /
fp32 accumulate.  N>1 (torchrun): one replica per GPU, no collective on the data path (inference shards by image) -> "weak".
Prints ONE JSON line on rank 0.  See DESIGN.md (Measurement) for the roofline arithmetic.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CFGS = {"s_psp": ("yolov5s_city_seg.yaml", 29.70e9), "m_lab": ("yolov5m_city_seg_lab.yaml", 80.27e9),
        "m_psp": ("yolov5m_city_seg.yaml", None), "s_bise": ("yolov5s_city_seg_bise.yaml", 32.91e9),
        "s_base": ("yolov5s_city_seg_base.yaml", 30.87e9)}
H, W = 512, 1024
# synthetic Detect objectness-bias shifts (per level) calibrated so that ~1% of the 32256 anchors pass obj>0.25
# (a realistic O(300) candidates/img NMS load instead of the ~10k the near-critical synthetic weights would give)
OBJ_BIAS_SHIFT = {"s_psp": (-17.5, -10.5, -18.2), "m_lab": (-5.9, -4.6, -5.2)}


def make_weights(tag):
    from multiyolov5_b200 import synth
    yml = CFGS[tag][0]
    cfg = synth.load_cfg(yml)
    sd = synth.synth_state_dict(synth.load_manifest(tag if tag in ("s_psp", "m_lab", "m_psp", "s_bise", "s_base") else "s_psp"), cfg, seed=1)
    no = cfg["nc"] + 5
    shifts = OBJ_BIAS_SHIFT.get(tag, (-10.0, -10.0, -10.0))
    for lvl in range(3):
        sd[f"model.25.m.{lvl}.bias"].view(-1, no)[:, 4] += shifts[lvl]
    return yml, cfg, sd


DUMP_LIMIT = 60 * 10 ** 6      # array bytes: with the .npy headers a dump stays under 64 MB


def dump_outputs(dirname, arrays):
    """writes each array as DIR/<name>.npy in float32, at most DUMP_LIMIT bytes of data.  An array that does not fit the remaining budget
    is replaced by a fixed seeded sample of its elements, and DIR/<name>_index.npy (float64) holds the flat positions taken."""
    os.makedirs(dirname, exist_ok=True)
    left = DUMP_LIMIT
    for name, a in sorted(arrays.items(), key=lambda kv: kv[1].size):
        a = np.asarray(a, np.float32)
        if a.nbytes > left:
            idx = np.sort(np.random.RandomState(0).choice(a.size, left // 12, replace=False)).astype(np.float64)   # 4 + 8 bytes each
            np.save(os.path.join(dirname, f"{name}_index.npy"), idx)
            a = a.reshape(-1)[idx.astype(np.int64)]
            left -= idx.nbytes
        np.save(os.path.join(dirname, f"{name}.npy"), a)
        left -= a.nbytes


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md 'clocks line')."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.stop_flag, self.samples = gpu_index, False, []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.gpu), "-lms", "20"],
                                 stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            return
        while not self.stop_flag:
            line = p.stdout.readline()
            if not line:
                break
            self.samples.append([s.strip() for s in line.split(",")])
        p.terminate()

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_reference_line(args, tag, steps, warmup, as_main):
    """the reference's CPU implementation of the path (oracle port: torch fp32 CPU + torchvision nms), one image per step."""
    from oracle import synth
    from oracle.cpu_pipeline import make_cpu_pipeline, reference_root
    yml, cfg, sd = make_weights(tag)
    x = synth.synth_image(1, H, W, seed=0)
    # the reference would run with torch's default (= all cores); small-batch convs often run faster with fewer threads, so give the
    # CPU arm its best case: probe a few thread counts and keep the fastest
    ncpu = os.cpu_count() or 1
    best = None
    for th in sorted({t for t in (8, 16, 32, 64, ncpu) if t <= ncpu}):
        pipe, kind = make_cpu_pipeline(cfg, sd, threads=th)
        pipe(x)
        t0 = time.perf_counter(); pipe(x); dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, th)
    pipe, kind = make_cpu_pipeline(cfg, sd, threads=best[1])
    for _ in range(warmup):
        pipe(x)
    ts, parts = [], []
    for _ in range(steps):
        t0 = time.perf_counter()
        _, _, tm = pipe(x)
        ts.append(time.perf_counter() - t0)
        parts.append(tm)
    med = float(np.median(ts))
    info = {"value": 1.0 / med, "unit": "images/s", "cores": pipe.threads, "kind": kind,
            "code": (f"unmodified reference tree at {reference_root()} (import-only stubs, oracle/ref_shims.py)" if kind == "reference" else
                     "oracle port of the detect.py job (oracle/cpu_pipeline.py): the reference is not an installable package and its tree is not on this box"),
            "sample": f"{steps} steps x 1 image 3x{H}x{W} fp32 (model {np.median([p['model'] for p in parts]) * 1e3:.1f} ms, nms "
                      f"{np.median([p['nms'] for p in parts]) * 1e3:.1f} ms, seg upsample+argmax {np.median([p['segpost'] for p in parts]) * 1e3:.1f} ms), "
                      f"os.cpu_count()={os.cpu_count()}, torch threads={pipe.threads} (fastest of 8/16/32/64/all)"}
    if not as_main:
        return info
    return {"metric": "images/sec @1024x512 (det+seg fwd)", "value": info["value"], "unit": "images/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": f"{yml} detect.py job (Model.forward + NMS 0.25/0.45 + seg upsample/argmax), 1x3x{H}x{W} per step on host CPU"},
            "cpu_baseline": info, "e2e": {"value": info["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def reference_gpu_infer(tag, B, steps, warmup):
    """detect.py job through torch's fp16 + cuDNN kernels on this GPU (oracle/gpu_pipeline.py): resident fp16 inputs, NROT batches > L2"""
    try:
        from oracle.gpu_pipeline import TorchHalfPipeline
        yml, cfg, sd = make_weights(tag)
        pipe = TorchHalfPipeline(cfg, sd)
        gen = torch.Generator(device="cuda").manual_seed(4321)
        xs = [torch.rand((B, 3, H, W), device="cuda", generator=gen).half() for _ in range(4)]
        for i in range(max(3, warmup)):
            pipe(xs[i % 4])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            pipe(xs[i % 4])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        e0.record()
        for i in range(steps):
            if pipe.model is not None:
                pipe.model(xs[i % 4])
            else:
                from oracle import restate
                with torch.no_grad():
                    restate.model_forward(cfg, pipe.sd, xs[i % 4], half=True)
        e1.record()
        torch.cuda.synchronize()
        ms_model = e0.elapsed_time(e1)
        return {"images_per_s": B * steps / (ms * 1e-3), "ms_per_step": ms / steps, "model_only_images_per_s": B * steps / (ms_model * 1e-3),
                "steps": steps, "kind": pipe.kind, "note": "python-loop NMS (torchvision.ops.nms per image) and per-image upsample+argmax as detect.py does"}
    except Exception as e:        # a baseline arm must never take the bench down
        return {"unavailable": f"{type(e).__name__}: {e}"[:300]}


def infer_record(tag, B, steps, warmup, world, min_seconds=1.0):
    """sub-record for another inference config (BASELINE.json configs[2]: yolov5m + Lab head, batch 8): same step as the headline"""
    import torch.distributed as dist
    from multiyolov5_b200.models.yolo import Model
    from multiyolov5_b200.utils.general import non_max_suppression, seg_argmax
    yml, cfg, sd = make_weights(tag)
    model = Model(yml)
    model.load_state_dict(sd)
    model.cuda().eval().half()
    gen = torch.Generator(device="cuda").manual_seed(99)
    xs = [torch.rand((B, 3, H, W), device="cuda", generator=gen).half() for _ in range(4)]

    def step(i):
        (z, _), seg = model(xs[i % 4])
        non_max_suppression(z, 0.25, 0.45, return_padded=True)
        seg_argmax(seg, (H, W))

    def run(n):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            step(i)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.barrier()
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    for i in range(max(3, warmup)):
        step(i)
    ms = run(steps)
    n_long = max(steps, int(min_seconds * 1e3 / (ms / steps)) + 1)
    ms_long = run(n_long)
    rec = {"workload": f"{yml} inference, batch {B}x3x{H}x{W} per GPU, half mode: Model.forward + NMS(0.25,0.45) + seg argmax", "n_gpus": world, "steps": steps,
           "ms_per_step": ms / steps, "images_per_s": B * world * steps / (ms * 1e-3),
           "sustained": {"steps": n_long, "seconds": ms_long * 1e-3, "images_per_s": B * world * n_long / (ms_long * 1e-3)},
           "gflop_per_image": (CFGS[tag][1] or 0) / 1e9}
    del model, xs
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--no-extras", action="store_true", help="skip the train / m_lab / reference-gpu sub-records (quick runs, ncu captures)")
    ap.add_argument("--cfg", default="s_psp", choices=list(CFGS))
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--fp32-logits", action="store_true", help="keep fp32 I/O (fp32 seg logits) instead of the reference's half() mode")
    ap.add_argument("--profile-ops", action="store_true", help="print the per-op device-time table to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (padded detections, their counts, the class map) as DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    warmup = max(args.warmup, 3)

    if args.impl == "reference":
        if rank == 0:
            print(json.dumps(cpu_reference_line(args, args.cfg, max(3, min(args.steps, 30)), min(warmup, 3), True)), flush=True)
        return
    if args.impl == "reference-gpu":
        # the reference's own GPU configuration (torch fp16 + cuDNN, cudnn.benchmark; detect.py:96-103,124) on ONE B200: a baseline arm
        if rank == 0:
            torch.cuda.set_device(local)
            B = args.batch or (16 if args.cfg.startswith("s_") else 8)
            rec = reference_gpu_infer(args.cfg, B, max(5, min(args.steps, 20)), warmup)
            line = {"metric": "images/sec @1024x512 (det+seg fwd)", "value": rec.get("images_per_s"), "unit": "images/s", "n_gpus": 1,
                    "steps": rec.get("steps"), "warmup": warmup, "ms_per_step": rec.get("ms_per_step"), "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": "f16 (torch / cuDNN)", "data": "synthetic", "impl": "reference-gpu",
                    "config": {"workload": f"{CFGS[args.cfg][0]} detect.py job, batch {B}x3x{H}x{W}, inputs resident in HBM"}, "detail": rec,
                    "gpu_launches": 0}
            print(json.dumps(line), flush=True)
        return

    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL prints its version banner on stdout when the communicator is created: keep stdout clean for the ONE JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    from multiyolov5_b200.models.yolo import Model
    from multiyolov5_b200.utils.general import non_max_suppression, seg_argmax
    tag = args.cfg
    B = args.batch or (16 if tag.startswith("s_") else 8)
    yml, cfg, sd = make_weights(tag)
    model = Model(yml)
    model.load_state_dict(sd)
    model.cuda().eval()
    if not args.fp32_logits:
        model.half()      # the reference's CUDA configuration (detect.py:96-103): fp16 parameters/IO -> seg logits come back as fp16
    eng = model.engine()

    # inputs: rotate over NROT different batches so that a step's input is never L2 resident from the previous step
    NROT = 4
    gen = torch.Generator(device="cuda").manual_seed(1234 + rank)
    xs_u8 = [torch.randint(0, 256, (B, 3, H, W), dtype=torch.uint8, device="cuda", generator=gen) for _ in range(NROT)]
    xs_f32 = [(x.float() / 255.0) if args.fp32_logits else (x.float() / 255.0).half() for x in xs_u8]
    host_u8 = [x.cpu().pin_memory() for x in xs_u8]

    # NMS (16 CTAs, latency bound) and the seg argmax (HBM bound) are independent consumers of the forward: run them concurrently
    s_nms = torch.cuda.Stream()
    ev_fwd, ev_nms = torch.cuda.Event(), torch.cuda.Event()

    def post(z, seg, cls_dtype=torch.int64):
        main = torch.cuda.current_stream()
        ev_fwd.record(main)
        with torch.cuda.stream(s_nms):
            s_nms.wait_event(ev_fwd)
            det, cnt = non_max_suppression(z, 0.25, 0.45, return_padded=True)
            ev_nms.record(s_nms)
        cls = seg_argmax(seg, (H, W), out_dtype=cls_dtype)
        main.wait_event(ev_nms)
        return det, cnt, cls

    def step_resident(i):
        (z, _raw), seg = model(xs_f32[i % NROT])
        return post(z, seg)

    # ---- end-to-end: pinned host uint8 frames -> device -> detections + class map -> pinned host, software-pipelined two deep
    # (copy-in stream / compute stream / copy-out stream, double-buffered device and host buffers; every step's H2D and D2H
    # happen inside the timed region).  The class map goes back as uint8 (19 classes); the reference moves the same map as int64.
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    dev_in2 = [torch.empty_like(xs_u8[0]) for _ in range(2)]
    host_cls2 = [torch.empty((B, H, W), dtype=torch.uint8).pin_memory() for _ in range(2)]
    host_det2 = [torch.empty((B, 300, 6), dtype=torch.float32).pin_memory() for _ in range(2)]
    host_cnt2 = [torch.empty((B,), dtype=torch.int32).pin_memory() for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_comp = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]
    keep = [None, None]

    def step_e2e(i):
        k = i % 2
        comp = torch.cuda.current_stream()
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_comp[k])                                    # compute(i-2) has consumed this input buffer
            dev_in2[k].copy_(host_u8[i % NROT], non_blocking=True)          # H2D: uint8 frames as detect.py:135
            ev_in[k].record(s_in)
        comp.wait_event(ev_in[k])
        comp.wait_event(ev_out[k])                                         # D2H(i-2) released the output slot
        (z, _raw), seg = model(dev_in2[k])                                 # /255 happens inside the first kernel (detect.py:137)
        det, cnt, cls = post(z, seg, torch.uint8)
        ev_comp[k].record(comp)
        keep[k] = (det, cnt, cls, seg, z)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_comp[k])
            host_det2[k].copy_(det, non_blocking=True)
            host_cnt2[k].copy_(cnt, non_blocking=True)
            host_cls2[k].copy_(cls, non_blocking=True)                     # D2H: class map as detect.py:193 (.cpu())
            ev_out[k].record(s_out)
        return det, cnt, cls

    def timed(fn, steps, sampler=None, finalize=None):
        if sampler:
            sampler.start()     # samples cover warm-up + timed region (identical load)
        for i in range(warmup + (40 if sampler else 0)):
            fn(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = None
        e0.record()
        for i in range(steps):
            fn(i)
        if finalize:
            finalize()       # e.g. make the timed stream wait for the last device->host copies
        e1.record()
        torch.cuda.synchronize()
        if sampler:
            sampler.stop_flag = True
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    last = {}

    def step_recorded(i):
        last["out"] = step_resident(i)

    sampler = ClockSampler(local) if rank == 0 else None
    ms_total = timed(step_recorded if args.dump_outputs else step_resident, args.steps, sampler)
    if args.dump_outputs and rank == 0:
        det, cnt, cls = (t.cpu().numpy() for t in last.pop("out"))      # timed() synchronised: these are the last timed step's results
        dump_outputs(args.dump_outputs, {"detections": det, "detection_counts": cnt, "class_map": cls})
    # the same step for >= 1 s (the driver's `steps` make a ~50 ms region: a burst figure; this one runs at sustained clocks / power)
    n_long = max(args.steps, int(1000.0 / (ms_total / args.steps)) + 1)
    sampler_long = ClockSampler(local) if rank == 0 else None
    if sampler_long:
        sampler_long.start()
    ms_long = timed(step_resident, n_long)
    if sampler_long:
        sampler_long.stop_flag = True
    det, cnt, cls = step_resident(0)
    torch.cuda.synchronize()
    n_cand = float(cnt.float().mean().item())
    launches_per_step = eng.launches() + 2 + 1          # forward ops + (nms filter, nms) + seg argmax
    def e2e_tail():
        for k in range(2):
            torch.cuda.current_stream().wait_event(ev_out[k])
    ms_e2e = timed(step_e2e, args.steps, finalize=e2e_tail)
    torch.cuda.synchronize()

    # ---- extra: from RAW camera frames (2048x1024 BGR uint8, pinned host) through the device-side letterbox/pre-process kernel
    # (SURVEY.md section 8f rank 1: replaces cv2.resize + transpose + /255 of utils/datasets.py:185-189 / detect.py:135-137);
    # same two-deep pipeline, H2D of 6.3 MB per frame inside the timed region
    from multiyolov5_b200.utils.datasets import preprocess
    RAW_H, RAW_W = 2 * H, 2 * W
    gen_raw = torch.Generator().manual_seed(4321 + rank)
    raw_host = [torch.randint(0, 256, (B, RAW_H, RAW_W, 3), dtype=torch.uint8, generator=gen_raw).pin_memory() for _ in range(2)]
    raw_dev = [torch.empty((B, RAW_H, RAW_W, 3), dtype=torch.uint8, device="cuda") for _ in range(2)]

    def step_raw(i):
        k = i % 2
        comp = torch.cuda.current_stream()
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_comp[k])
            raw_dev[k].copy_(raw_host[k], non_blocking=True)
            ev_in[k].record(s_in)
        comp.wait_event(ev_in[k])
        comp.wait_event(ev_out[k])
        x, _, _ = preprocess(raw_dev[k], (H, W), stride=32, half=not args.fp32_logits)
        (z, _raw), seg = model(x)
        det, cnt, cls = post(z, seg, torch.uint8)
        ev_comp[k].record(comp)
        keep[k] = (det, cnt, cls, seg, z, x)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_comp[k])
            host_det2[k].copy_(det, non_blocking=True)
            host_cnt2[k].copy_(cnt, non_blocking=True)
            host_cls2[k].copy_(cls, non_blocking=True)
            ev_out[k].record(s_out)
    ms_raw = timed(step_raw, args.steps, finalize=e2e_tail)
    torch.cuda.synchronize()
    del raw_dev, raw_host

    # model-only and fused variants (reported as extras)
    def step_model(i):
        model(xs_f32[i % NROT])
    ms_model = timed(step_model, args.steps)

    def step_fused(i):
        out = model(xs_f32[i % NROT], seg_argmax=True)
        non_max_suppression(out[0][0], 0.25, 0.45, return_padded=True)
    ms_fused = timed(step_fused, args.steps)

    # per-op device time (CUDA events around every op on the launching stream) -> roofline of the tcgen05 conv kernel
    roof = None
    if rank == 0:
        reps = 5
        acc = None
        for r in range(reps + 2):
            eng.forward(xs_f32[r % NROT], profile=True)
            if r >= 2:
                acc = np.array(eng.last_profile) if acc is None else acc + np.array(eng.last_profile)
        per_op = acc / reps
        pb = eng.last_plan.pb
        from multiyolov5_b200 import _lib
        import ctypes as C
        from multiyolov5_b200.plan import conv_algorithmic_flops
        conv_ms = simt_ms = 0.0
        n_conv = n_simt = 0
        flops = simt_flops = 0.0
        info = (C.c_int32 * 12)()
        conv_table = []
        layer_rows = []
        for i, o in enumerate(pb.ops):
            if o.kind == _lib.OP_CONV:
                s = pb.slots[o.slot].conv
                f = conv_algorithmic_flops(s, B, o.out)      # the reference layer's 2 x MACs (restated layer-0 conv included)
                _lib.check(_lib.lib().myolo_plan_conv_info(eng.last_plan.handle, i, info))
                if info[0]:      # tcgen05 kernel
                    conv_ms += per_op[i]; n_conv += 1; flops += f
                    # algorithmic bytes of the launch: input + output (+ residual) activations once, weights once, fp16 (fp32 head outputs: 4 B)
                    nbytes = (B * o.in_.h * o.in_.w * o.in_.c * 2 + B * o.out.h * o.out.w * s.out_channels * (2 if o.out.buf.dtype == _lib.F16 else 4)
                              + (B * o.out.h * o.out.w * s.out_channels * 2 if o.in2 is not None else 0)
                              + s.out_channels * s.in_channels * s.kernel_size[0] * s.kernel_size[1] * 2)
                    layer_rows.append((f, nbytes, per_op[i]))
                else:            # CUDA-core kernel (maps < one 128-pixel tile: PPM bins, FFM attention FCs)
                    simt_ms += per_op[i]; n_simt += 1; simt_flops += f
                conv_table.append((i, o.tag, f"{s.in_channels}->{s.out_channels} k{s.kernel_size[0]}s{s.stride[0]}d{s.dilation[0]} @{o.out.h}x{o.out.w}",
                                   list(info), per_op[i] * 1e3, f))
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        ach = flops / (conv_ms * 1e-3) / 1e12
        traffic = None
        try:   # dram__bytes_read+write per conv_tc launch from the committed `ncu --set full` capture of the same step (profiles/)
            tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            if tj.get("cfg") == tag and tj.get("batch") == B:
                traffic = tj["dram_bytes_per_launch"]
        except Exception:
            pass
        roof = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": traffic,
                "kernel": "conv_tc_kernel (the tcgen05 Conv+BN+SiLU launches of one forward; CUDA-core conv launches are listed separately)",
                "launches": n_conv, "avg_launch_ms": conv_ms / n_conv, "simt_conv_launches": n_simt, "simt_conv_ms": simt_ms,
                "simt_conv_flops_per_step": simt_flops,
                "algorithmic_flops_per_step": flops, "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PF sustained",
                "conv_share_of_forward": conv_ms / float(per_op.sum())}
        # the same launches against their OWN roofline min(tensor, AI x HBM): most layers of this network are activation-bandwidth bound
        # (1x1 convs, 16-64 channel layers), so the aggregate tensor fraction above cannot approach 1 whatever the kernel does
        hbm_peak = peaks.get("hbm_gbs", 6500.0) * 1e9
        t_bound = [max(f / (peak * 1e12), nb / hbm_peak) * 1e3 for f, nb, _ in layer_rows]
        roof["per_layer"] = {"bound_ms": float(sum(t_bound)), "measured_ms": float(conv_ms), "frac": float(sum(t_bound) / conv_ms),
                             "hbm_bound_launches": int(sum(1 for (f, nb, _) in layer_rows if nb / hbm_peak > f / (peak * 1e12))),
                             "tensor_bound_launches": int(sum(1 for (f, nb, _) in layer_rows if nb / hbm_peak <= f / (peak * 1e12))),
                             "note": "sum over the tcgen05 conv launches of max(FLOP / tensor peak, algorithmic bytes / HBM peak) / measured device time"}
        if args.profile_ops:
            for i, o in enumerate(pb.ops):
                print(f"{i:3d} kind={o.kind:2d} {o.tag:24s} {per_op[i] * 1e3:9.1f} us", file=sys.stderr)
            print("# conv launches: op, layer, shape, [tc, grid, smem, BN, stages, mode, ws, G, tiles, ntn, kc, cta/sm], us, TFLOP/s", file=sys.stderr)
            for (i, tg, shp, inf, us, f) in conv_table:
                print(f"#conv {i:3d} {tg:16s} {shp:30s} {inf} {us:8.1f} us {f / (us * 1e-6) / 1e12:7.1f} TF/s", file=sys.stderr)

    if rank == 0:
        imgs = B * world * args.steps
        line = {"metric": "images/sec @1024x512 (det+seg fwd)", "value": imgs / (ms_total * 1e-3), "unit": "images/s", "n_gpus": world,
                "steps": args.steps, "warmup": warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f16 storage / f32 accumulate", "data": "synthetic",
                "config": {"workload": f"{yml} inference, batch {B}x3x{H}x{W} per GPU: Model.forward (z, raw, {'fp32' if args.fp32_logits else 'fp16'} seg logits) + NMS(0.25,0.45) + "
                                       "seg upsample/argmax", "global_batch": B * world, "parallelism": f"replicas x{world} (no collective)",
                           "l2": f"inputs rotate over {NROT} batches ({NROT * B * 3 * H * W * 4 / 1e6:.0f} MB > 126 MB L2); activations are rewritten every step",
                           "nms_candidates_kept_per_img": n_cand},
                "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": "images/s", "h2d_bytes_per_step": B * 3 * H * W,
                        "d2h_bytes_per_step": B * H * W * 1 + B * 300 * 6 * 4 + B * 4,
                        "note": "2-deep software pipeline over 3 streams; class map returned as uint8"},
                "gpu_launches": launches_per_step * args.steps,
                "e2e_from_raw_frames": {"value": imgs / (ms_raw * 1e-3), "unit": "images/s", "h2d_bytes_per_step": B * 4 * H * W * 3,
                                        "note": "2048x1024 BGR uint8 frames -> device letterbox/pre-process kernel (bit exact with cv2) -> forward -> post-process"},
                "model_only_images_per_s": imgs / (ms_model * 1e-3), "fused_argmax_images_per_s": imgs / (ms_fused * 1e-3),
                "clocks": sampler.summary() if sampler else None, "roofline": roof,
                "sustained": {"steps": n_long, "seconds": ms_long * 1e-3, "ms_per_step": ms_long / n_long,
                              "value": B * world * n_long / (ms_long * 1e-3), "clocks": sampler_long.summary() if sampler_long else None,
                              "note": "same resident step as `value`, timed for >= 1 s"}}
        line["e2e"]["d2h_note"] = "class map returned as uint8 (19 classes); the reference's .cpu() moves the same map as int64, 8x the bytes"
    # ---- sub-records for the other BASELINE.json configs (every rank takes part: the train step contains the path's one collective)
    extras = {}
    if not args.no_extras and tag == "s_psp" and args.batch is None:
        del xs_u8, xs_f32, dev_in2, keep
        model = eng = None
        torch.cuda.empty_cache()
        from tools.bench_train import train_record
        extras["train"] = train_record(world, rank, steps=max(6, args.steps // 2), warmup=warmup, B=4, with_reference_gpu=(world == 1))
        extras["m_lab"] = infer_record("m_lab", 8, args.steps, warmup, world)
        if rank == 0 and world == 1:
            extras["reference_gpu"] = reference_gpu_infer(tag, B, 10, warmup)
    if rank == 0:
        line.update(extras)
        if "reference_gpu" in extras and extras["reference_gpu"].get("images_per_s"):
            line["reference_gpu"]["ours_over_torch"] = line["value"] / extras["reference_gpu"]["images_per_s"]
        if "train" in extras and isinstance(extras["train"].get("reference_gpu"), dict) and extras["train"]["reference_gpu"].get("ms_per_step"):
            extras["train"]["reference_gpu"]["ours_over_torch"] = extras["train"]["reference_gpu"]["ms_per_step"] / extras["train"]["ms_per_step"]
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_reference_line(args, tag, 8, 2, False)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
