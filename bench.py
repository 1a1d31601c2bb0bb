#!/usr/bin/env python
"""bench.py -- FuseTrack frame pairs / second on synthetic 1024x2048 pairs (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU, clips sharded)
  python bench.py --impl reference --gpus N --steps K ...  # reference arm: the oracle port on the host CPU cores

One step = one `simple_test` call = one frame pair -> one panoptic frame.  Prints ONE JSON line (rank 0).
The headline (`value`, `e2e`, `roofline`) is measured in the PARITY precision "tc32" (fp32 activations, tcgen05 with split
fp16 operands: label maps / ids identical to the oracle, tests/test_gpu_e2e.py, tests/test_gpu_fullsize.py); the bf16
fast mode (one tensor-core pass, ~0.99 label agreement) is timed in the same run and reported under `fast_mode`.
  value      : pairs/s over ONE device-timed region (CUDA events) of K steps through the public clip loop
               (vps_b200.runner.ClipRunner), inputs already resident in HBM, max over ranks, summed over ranks
  --workload viper : BASELINE config 4 -- 30-frame 1088x1920 clips (1080 padded to 1088), one clip stream per GPU
  e2e        : the same region with HOST (pinned) frames: H2D of both frames and D2H of the label maps of every step
               inside the timed region
  sequential_ms_per_pair : one pair at a time, L2 flushed in between (latency)
  next_rows  : the first rows past the hot path (SURVEY 8f): unified pan result, VPQ frame confusion
  roofline   : the dominant kernel (tcgen05 implicit-GEMM conv, all launches of a step): algorithmic conv FLOPs /
               summed kernel time, against the measured cuBLAS bf16 peak of MEASURED_PEAKS.json
  cpu_baseline: the oracle (CPU port of the reference math) on a bounded sample, host cores
  --dump-outputs DIR : after the timed steps, the results of the last step of the `value` region as DIR/<name>.npy
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

H_FULL, W_FULL = 1024, 2048
METRIC = "FuseTrack frame pairs/s on synthetic 1024x2048 pairs"
# algorithmic dense work per pair at 1024x2048 (BASELINE.md section 2, SURVEY 8d), GFLOP
GFLOP_R50FPN_PAIR = 1158.4
GFLOP_ALL_PAIR = 5017.0


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu=0):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag = gpu, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def synth_pairs(n, H, W, seed=0):
    """n distinct synthetic (img, ref) pairs, post-Normalize statistics, ref = shifted img + noise (SURVEY 8d)."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for i in range(n):
        img = torch.randn(1, 3, H, W, generator=g)
        ref = torch.roll(img, shifts=(2 + i % 3, 3 + i % 5), dims=(2, 3)) + 0.05 * torch.randn(1, 3, H, W, generator=g)
        out.append((img.contiguous(), ref.contiguous()))
    return out


def meta(iid, H, W):
    return dict(filename="synthetic_city_%06d.png" % iid, iid=iid, img_shape=(H, W, 3), pad_shape=(H, W, 3),
                ori_shape=(H, W, 3), scale_factor=1.0)


def _sample(t, k, seed):
    """t itself, or k of its elements at seeded random flat positions when it has more"""
    if t.numel() <= k:
        return t
    idx = torch.randint(t.numel(), (k,), generator=torch.Generator().manual_seed(seed))
    return t.reshape(-1)[idx.to(t.device)]


def result_arrays(r):
    """the arrays a caller of the timed path receives for one pair (bbox_results, segm_results, pano_results), as
    float32 / float64 numpy arrays, at most ~34 MB in all: label maps up to 4M pixels whole (a seeded sample beyond),
    a seeded 64K-element sample of each FPN level.  Copied at once: the runner reuses its output buffers."""
    bbox, _, pano = r
    ids = sorted(bbox)
    out = {"bbox_ids": np.array(ids, np.float64),
           "bbox_labels": np.array([bbox[i]["label"] for i in ids], np.float64),
           "bbox": np.array([bbox[i]["bbox"] for i in ids], np.float32).reshape(-1, 4)}
    for name in ("panoptic_outputs", "fcn_outputs"):
        out[name] = _sample(pano[name], 1 << 22, 0).cpu().numpy().astype(np.float32)
    for name in ("panoptic_cls_inds", "panoptic_det_labels", "panoptic_det_obj_ids"):
        out[name] = pano[name].cpu().numpy().astype(np.float64)
    out["panoptic_cls_prob"] = pano["panoptic_cls_prob"].cpu().numpy().astype(np.float32)
    for lvl, f in enumerate(pano["fpn_feats"]):
        out["fpn_feats_%d_sample" % lvl] = _sample(f.float(), 1 << 16, 1 + lvl).cpu().numpy()
    return out


# ------------------------------------------------------------------------------------------------ CPU arms
def oracle_model():
    from oracle.model import PanopticFuseTrack as Oracle
    from vps_b200.synth import make_weights
    m = Oracle()
    make_weights(m, "C", 0)
    return m


def host_threads():
    """threads used for the CPU arms: all cores up to 32 (beyond that torch's CPU convolutions stop scaling on the
    small per-op work of a frame pair and oversubscription makes them slower)."""
    return max(1, min(os.cpu_count() or 1, 32))


def time_oracle(model, H, W, reps, threads):
    torch.set_num_threads(threads)
    pairs = synth_pairs(1, H, W, seed=3)
    times = []
    for r in range(reps):
        t = time.perf_counter()
        model.simple_test(pairs[0][0], dict(iid=10001 + r, img_shape=(H, W, 3)), pairs[0][1])
        times.append(time.perf_counter() - t)
    return times


# The CPU arms time the oracle on ONE fixed sample size (deterministic from run to run): a 512x1024 pair = 1/4 of the
# 1024x2048 area, ~5-10 s per pair on 32 host threads, scaled by area (the dense work is linear in pixels; the fixed
# per-frame head cost makes the sample slightly pessimistic for the CPU).  VPS_BENCH_CPU_SAMPLE=HxW overrides it
# (1024x2048 = the full workload, ~30-40 s per pair).
def cpu_sample():
    v = os.environ.get("VPS_BENCH_CPU_SAMPLE", "512x1024").lower().split("x")
    return int(v[0]), int(v[1])


def cpu_baseline():
    """Oracle on the host cores on the fixed bounded sample: 1 warm-up + 2 timed pairs."""
    threads = host_threads()
    m = oracle_model()
    Hs, Ws = cpu_sample()
    frac = Hs * Ws / float(H_FULL * W_FULL)
    time_oracle(m, 64, 128, 1, threads)
    ts = time_oracle(m, Hs, Ws, 3, threads)[1:]
    t = float(np.mean(ts))
    return {"value": frac / t, "unit": "pairs/s (1024x2048-equivalent)", "cores": threads, "kind": "port",
            "sample": "oracle simple_test, 2 timed pairs at %dx%d (%.3g of the 1024x2048 area) in %.2f s each, scaled by area; "
                      "fp32, torch CPU ops" % (Hs, Ws, frac, t)}


def run_reference_arm(args):
    """--impl reference: the reference's own math on the host CPU.  The reference cannot execute on this stack
    (mmcv 0.2.14 + THC extensions, hard .cuda() calls; DESIGN.md), so this is the oracle port (kind 'port').
    Each step = one frame pair at a bounded sample size chosen so that a step takes a few seconds."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:            # no process group is created in this arm: the other ranks have nothing to do and exit at once
        return
    threads = host_threads()
    m = oracle_model()
    Hs, Ws = cpu_sample()
    frac = Hs * Ws / float(H_FULL * W_FULL)
    time_oracle(m, 64, 128, 1, threads)                           # lazy inits
    times = time_oracle(m, Hs, Ws, args.warmup + args.steps, threads)[args.warmup:]
    t = float(np.mean(times))
    v = frac / t
    sample = "each step = one %dx%d pair (%.3g of the 1024x2048 area) on %d CPU threads, scaled by area" % (Hs, Ws, frac, threads)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t / frac, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "FuseTrack inference, synthetic 2-frame 1024x2048 pair, random-init (synthetic set C) weights (CPU arm: fixed bounded sample, see `sample`)",
                       "sample": sample},
            "cpu_baseline": {"value": v, "unit": "pairs/s (1024x2048-equivalent)", "cores": threads, "kind": "port",
                             "sample": "oracle simple_test, %d steps; %s" % (args.steps, sample)},
            "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm
def build_product(precision, device):
    from vps_b200 import ConfigDict, build_detector, fusetrack_cfg
    from vps_b200.synth import make_weights
    c = fusetrack_cfg()
    det = build_detector(ConfigDict(c["model"]), train_cfg=None, test_cfg=ConfigDict(c["test_cfg"]))
    make_weights(det, "C", 0)
    det.precision = precision
    det = det.to(device)
    det.prepare()
    return det


def stock_pytorch_r50fpn(dev, H, W, flush):
    """Context (BASELINE.md section 3 / SURVEY 8d "the real bar to beat"): the SAME ResNet-50-FPN math as stock PyTorch
    modules (the oracle's, i.e. test infrastructure -- not the product) on this GPU through cuDNN: fp32 (TF32 off), TF32 and
    bf16 channels_last autocast, both frames as a batch of 2, median of 5 with L2 flush."""
    from oracle.model import PanopticFuseTrack as Oracle
    from vps_b200.synth import make_weights
    m = Oracle()
    make_weights(m, "C", 0)
    net = torch.nn.Sequential()
    bb, neck = m.backbone.to(dev).eval(), m.neck.to(dev).eval()
    x = torch.randn(2, 3, H, W, device=dev)
    out = {}

    def run(tag, xin, ctx):
        with torch.no_grad(), ctx:
            for _ in range(2):
                neck(bb(xin))
            torch.cuda.synchronize()
            ts = []
            for i in range(5):
                flush.fill_(i)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); neck(bb(xin)); b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
        ms = sorted(ts)[2]
        out[tag] = {"ms": round(ms, 3), "tflops": round(GFLOP_R50FPN_PAIR * (H * W) / float(H_FULL * W_FULL) / ms, 1)}

    import contextlib
    torch.backends.cudnn.benchmark = True
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    run("fp32", x, contextlib.nullcontext())
    torch.backends.cudnn.allow_tf32 = True
    run("tf32", x, contextlib.nullcontext())
    bb.to(memory_format=torch.channels_last); neck.to(memory_format=torch.channels_last)
    run("bf16_channels_last", x.contiguous(memory_format=torch.channels_last), torch.autocast("cuda", dtype=torch.bfloat16))
    out["what"] = "oracle ResNet-50 + FPN modules (stock torch.nn / cuDNN, eager), 2 frames %dx%d as one batch; algorithmic 1158.4 GFLOP" % (H, W)
    return out


def run_gpu_arm(args):
    from vps_b200 import ops
    from vps_b200 import parallel as P
    rank, local, world = P.env_world()
    # the CPU leg (rank 0, N = 1 only) runs BEFORE the process group exists: no GPU spins in a collective meanwhile
    cpu_leg = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_leg = cpu_baseline()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    P.init("nccl", dev)
    viper = args.workload == "viper"
    H, W = (1088, 1920) if viper else (args.height, args.width)
    det = build_product(args.precision, dev)
    det.label_dtype = torch.uint8                    # the reference's collector casts both maps to uint8 (test_vpq.py:52-56)
    NPAIR = 4                                        # 4 distinct pairs = 201 MB of fp32 frames (> 126 MB L2)
    host = [(a.pin_memory(), b.pin_memory()) for a, b in synth_pairs(NPAIR, H, W, seed=100 + rank)]
    devp = [(a.to(dev), b.to(dev)) for a, b in host]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    CLIP = 30                                        # clip length (Cityscapes-VPS and the VIPER workload): tracker memory resets

    def step(i):
        iid = 10000 * (1 + rank) + 1 + (i % CLIP)
        a, b = devp[i % NPAIR]
        return det.simple_test(a, [meta(iid, H, W)], ref_img=[b])

    def timed(nsteps, offset):
        evs = []
        for i in range(nsteps):
            flush.fill_(i & 0xff)                    # L2 flush between timed iterations (outside the timed span)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            step(offset + i)
            e.record()
            evs.append((s, e))
        torch.cuda.synchronize()
        return [s.elapsed_time(e) for s, e in evs]

    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    # ---- the clip loop a user runs (vps_b200.runner.ClipRunner = single_gpu_test of tools/test_vpq.py): the static part
    # of pair i+1 (CUDA graph, second instance) is enqueued before pair i's data-dependent tail, uploads / downloads ride
    # a copy stream.  ONE timed region over all K steps; `value` takes the frames from HBM, `e2e` from pinned host memory.
    from vps_b200.runner import ClipRunner
    # viper: streaming clips -- the reference frame of frame t is frame t - 1 (cityscapes_vps.py:137-142), so the runner
    # reuses the previous pair's FPN features as reference features (results bit-identical: tests/test_gpu_e2e.py)
    runner = ClipRunner(det, dev, streaming=viper)
    last = {}                                        # the most recent result a region yielded

    def region(n, offset, resident):
        src = devp if resident else host
        if viper:       # a chain: frame k of the clip is src[k % NPAIR][0]; the first frame of a clip references itself
            def chain():
                for i in range(n):
                    k = (offset + i) % CLIP
                    cur = src[(offset + i) % NPAIR][0]
                    yield (cur, cur if k == 0 else src[(offset + i - 1) % NPAIR][0])
            pairs = chain()
        else:
            pairs = (src[(offset + i) % NPAIR] for i in range(n))
        metas = (meta(10000 * (1 + rank) + 1 + ((offset + i) % CLIP), H, W) for i in range(n))
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        chk = 0
        for r in runner.run(pairs, metas, resident=resident):
            chk += int(r[2]["panoptic_outputs"][0, 0, 0])       # the maps are host tensors here
            last["r"] = r
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e)

    # untimed: every CUDA-graph instance the timed regions replay must exist (2 ping-pong slots x {cached, uncached reference
    # features} in the streaming workload: each needs a warm call and a capturing call), pinned buffers allocated
    for _ in range(2 if viper else 1):
        region(max(args.warmup, 6), args.warmup, True)
        region(4 if viper else 2, args.warmup, False)
    torch.cuda.synchronize()
    P.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = ops.launch_count()
    ms = [region(args.steps, args.warmup + 5, True)]
    launches = ops.launch_count() - l0
    dump = result_arrays(last["r"]) if args.dump_outputs and rank == 0 else None
    torch.cuda.synchronize()
    P.barrier()
    ms_e2e = [region(args.steps, args.warmup + 5 + args.steps, False)]
    # host link check: the e2e region needs 50 MB of H2D per pair; a slow link (NUMA-remote pinned memory, shared PCIe)
    # bounds e2e below `value` and shows up here
    hs, he = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    hs.record()
    for i in range(4):
        host[i % NPAIR][0].to(dev, non_blocking=True)
        host[i % NPAIR][1].to(dev, non_blocking=True)
    he.record()
    torch.cuda.synchronize()
    h2d_gbps = 8 * 3 * H * W * 4 / (hs.elapsed_time(he) * 1e-3) / 1e9
    sampler.stop_flag = True
    seq_ms = timed(min(args.steps, 5), args.warmup)               # one pair at a time, L2 flushed: latency of a pair
    # ---- the bf16 fast mode (one tensor-core pass; NOT the reference's precision) in the same run, same regions
    fast = None
    if args.precision == "tc32" and not args.no_fast_mode:
        det.precision = "bf16"
        for i in range(3):
            step(i)
        region(5, 0, True)
        region(2, 0, False)
        torch.cuda.synchronize()
        P.barrier()
        f_ms = region(args.steps, args.warmup + 5, True)
        P.barrier()
        f_e2e = region(args.steps, args.warmup + 5 + args.steps, False)
        f_dev, f_e = [v / 1e3 for v in P.max_over_ranks([f_ms, f_e2e], dev)]
        fast = {"precision": "bf16", "value": world * args.steps / f_dev, "e2e": world * args.steps / f_e, "unit": "pairs/s",
                "ms_per_step": 1e3 * f_dev / args.steps,
                "parity": "bf16 operands, one tcgen05 pass: label agreement with the oracle 0.99 (semantic 0.9945 / panoptic 0.9896 "
                          "at 1024x2048, tests/test_gpu_fullsize.py) -- lower precision than the reference, reported for context"}
        det.precision = args.precision
    # ---- SURVEY 8f rank 1 (the step after the path): get_unified_pan_result on the GPU, timed alone on a real result
    from vps_b200.postproc import PanUnifier
    unifier = PanUnifier()
    r_last = step(args.warmup)
    u_args = (r_last[2]["fcn_outputs"], r_last[2]["panoptic_outputs"], r_last[2]["host"]["panoptic_cls_inds"],
              r_last[2]["host"]["panoptic_det_obj_ids"])
    unifier(*u_args)
    torch.cuda.synchronize()
    u_evs = []
    for i in range(10):
        flush.fill_(i)
        a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a_.record(); unifier(*u_args); b_.record()
        u_evs.append((a_, b_))
    torch.cuda.synchronize()
    unify_us = 1e3 * float(np.median([a_.elapsed_time(b_) for a_, b_ in u_evs]))
    unify_bytes = H * W * (3 * det.label_dtype.itemsize + 3)      # seg + pan read, pan re-read, 3 channels written
    # ---- SURVEY 8f rank 2: the pixel-level step of the VPQ evaluator (np.unique over 64-bit (gt, pred) codes of a frame)
    from vps_b200 import vpq as VPQ
    rs = np.random.default_rng(0)
    gt_np = (rs.integers(0, 40, size=(H // 16, W // 16)).repeat(16, 0).repeat(16, 1) * 1000 + 7).astype(np.int64)
    pr_np = (rs.integers(0, 60, size=(H // 8, W // 8)).repeat(8, 0).repeat(8, 1) * 997).astype(np.int64)
    gt_d, pr_d = torch.from_numpy(gt_np).to(dev), torch.from_numpy(pr_np).to(dev)
    VPQ.frame_confusion(gt_d, pr_d)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(5):
        VPQ.frame_confusion(gt_d, pr_d)                           # includes the read-back of the table (it syncs)
    conf_us = (time.perf_counter() - t0) / 5 * 1e6
    t0 = time.perf_counter()
    np.unique(gt_np.astype(np.uint64) * np.uint64(VPQ.OFFSET) + pr_np.astype(np.uint64), return_counts=True)
    conf_cpu_us = (time.perf_counter() - t0) * 1e6
    t_dev, t_e2e = [v / 1e3 for v in P.max_over_ranks([sum(ms), sum(ms_e2e)], dev)]     # max over ranks
    value = world * args.steps / t_dev
    e2e = world * args.steps / t_e2e

    # ---- per-kernel attribution (separate instrumented steps, not part of the timed region)
    roof, breakdown = None, None
    if rank == 0:
        ops.PROFILE = []
        for i in range(2):
            step(args.warmup + 2 * args.steps + i)
        torch.cuda.synchronize()
        rec, ops.PROFILE = ops.PROFILE, None
        if args.profile_out:
            os.makedirs(os.path.dirname(os.path.abspath(args.profile_out)) or ".", exist_ok=True)
            with open(args.profile_out, "w") as f:
                for name, s, e, fl, tag, scope in rec[len(rec) // 2:]:
                    f.write(json.dumps({"fn": name, "ms": s.elapsed_time(e), "flops": fl, "tag": tag, "scope": scope}) + "\n")
        agg, scopes = {}, {}
        for name, s, e, fl, tag, scope in rec:
            sc = scopes.setdefault(scope, [0.0, 0.0])
            sc[0] += s.elapsed_time(e) / 2; sc[1] += fl / 2
        for name, s, e, fl, tag, scope in rec:
            a = agg.setdefault(name, [0.0, 0.0, 0])
            a[0] += s.elapsed_time(e); a[1] += fl; a[2] += 1
        tc_ms, tc_fl, tc_n = 0.0, 0.0, 0
        tc32 = args.precision == "tc32"
        names = ("vps_conv2d_tc32", "vps_conv2d_tc32_multi", "vps_deform_conv_tc32") if tc32 else \
                ("vps_conv2d_tc", "vps_conv2d_tc_multi", "vps_deform_conv_tc")
        for kname in names:
            a_ = agg.get(kname, [0.0, 0.0, 0])
            tc_ms, tc_fl, tc_n = tc_ms + a_[0], tc_fl + a_[1], tc_n + a_[2]
        pk = peaks()
        if tc_ms > 0:
            ach = tc_fl / (tc_ms * 1e-3) / 1e12
            passes = 3 if tc32 else 1
            # DRAM traffic of the same kernels over one step, from the committed ncu pass (profiles/, see its README)
            traffic = None
            tp = os.path.join(ROOT, "profiles", "r2_dram_traffic.json")
            if os.path.exists(tp):
                try:
                    traffic = json.load(open(tp)).get("tc32" if tc32 else "bf16")
                except Exception:
                    traffic = None
            roof = {"bound": "tensor",
                    "kernel": ("conv_igemm_tc32_kernel + dcn_igemm_tc32_kernel" if tc32 else "conv_igemm_tc_kernel + dcn_igemm_tc_kernel")
                              + " (all %d launches of a step)" % (tc_n // 2),
                    "achieved": ach, "peak": pk["tf_sus"], "unit": "TFLOP/s", "frac": ach / pk["tf_sus"], "traffic": traffic,
                    "peak_source": pk["src"] + " bf16_tflops_sustained (cuBLAS bf16, back to back)",
                    "flops_per_step": tc_fl / 2, "ms_per_step": tc_ms / 2,
                    "tensor_passes": passes,
                    "tensor_pipe_frac": passes * ach / pk["tf_sus"],
                    "note": "achieved = ALGORITHMIC conv FLOPs (2*MAC of the fp32 layer) / summed kernel time; the parity precision "
                            "executes 3 f16 tensor-core products per algorithmic MAC (fp16 value + scaled residual split of both "
                            "operands), so frac <= 1/3 by construction and tensor_pipe_frac = 3 * frac is the pipe utilisation"
                            if tc32 else "achieved = algorithmic conv FLOPs / summed kernel time"}
        total_ms = sum(a[0] for a in agg.values())
        breakdown = {k: {"ms_per_step": round(a[0] / 2, 3), "share": round(a[0] / total_ms, 4), "calls": a[2] // 2}
                     for k, a in sorted(agg.items(), key=lambda kv: -kv[1][0])[:12]}

    if rank == 0:
        clocks = sampler.summary()
        bytes_in = 2 * 3 * H * W * 4
        bytes_out = 2 * H * W * det.label_dtype.itemsize
        line = {"metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * t_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"tc32": "f32 (tcgen05: 3 split-f16 products per MAC, fp32 accumulate promoted to RN register sums)",
                          "bf16": "bf16", "fp32": "f32 (CUDA cores)"}[args.precision], "data": "synthetic",
                "config": {"workload": ("VIPER-shape streaming inference, synthetic 30-frame 1088x1920 clips (1080 padded to 1088), " if viper else
                                        "FuseTrack inference, synthetic 2-frame %dx%d pair, " % (H, W)) +
                                       "random-init (synthetic set C) weights, 1 clip stream per GPU",
                           "precision": args.precision,
                           "ref_feature_cache": ("on: frame t's FPN features are reused as the reference features of frame t+1 "
                                                 "(one ResNet-50-FPN pass per pair; algorithmic FLOPs still counted on the reference's "
                                                 "two-pass basis)") if viper else "off (independent pairs)",
                           "parallelism": "clip-sharded replicas x%d, no data-path collective" % world,
                           "l2": "4 rotating input pairs (201 MB of fp32 frames > 126 MB L2) in both timed regions, steps are "
                                 "pipelined so no flush between them; sequential_ms_per_pair flushes 256 MiB between pairs",
                           "pipelining": "static part of pair i+1 (second CUDA-graph instance, side stream) overlaps pair i's "
                                         "tracker/mask/fusion tail; max(W,5) + 2 untimed runner steps precede the timed regions",
                           "labels": "uint8 label maps (same values as the reference's int64; its collector casts to uint8)",
                           "precision_note": "tc32 = the parity precision (label maps / ids identical to the oracle: tests/test_gpu_e2e.py, "
                                             "tests/test_gpu_fullsize.py); --precision bf16 = fast mode, --precision fp32 = CUDA-core debugging twin"},
                "e2e": {"value": e2e, "unit": "pairs/s", "h2d_bytes_per_step": bytes_in, "d2h_bytes_per_step": bytes_out,
                        "h2d_gbps_measured": round(h2d_gbps, 2)},
                "gpu_launches": int(launches), "clocks": clocks,
                "sequential_ms_per_pair": float(np.median(seq_ms)),
                "next_rows": {"unify_pan": {"what": "get_unified_pan_result on the GPU (SURVEY 8f rank 1), one 1024x2048 frame, "
                                                    "host-side id bookkeeping + 3 kernels, L2 flushed",
                                            "us_per_frame": round(unify_us, 1), "algorithmic_bytes": unify_bytes,
                                            "hbm_gbps": round(unify_bytes / (unify_us * 1e-6) / 1e9, 1),
                                            "hbm_frac": round(unify_bytes / (unify_us * 1e-6) / 1e9 / peaks()["hbm"], 4)},
                              "vpq_frame_confusion": {"what": "np.unique over (gt, pred) codes of one 1024x2048 frame (SURVEY 8f rank 2): "
                                                              "pack + 64-bit radix sort + run-length encode + table read-back",
                                                      "us_per_frame": round(conf_us, 1), "numpy_us_per_frame": round(conf_cpu_us, 1)}},
                "conv_flop_frac_whole_path": GFLOP_ALL_PAIR * (H * W) / float(H_FULL * W_FULL) * 1e9 * args.steps / t_dev / 1e12 / peaks()["tf_sus"]}
        if roof:
            line["roofline"] = roof
        if breakdown:
            line["breakdown"] = breakdown
            line["stages"] = {k: {"ms": round(v[0], 3), "gflop": round(v[1] / 1e9, 1)} for k, v in scopes.items()}
            if "r50fpn" in scopes:      # north-star target: fraction of the conv-FLOP roofline on 2 x ResNet-50-FPN
                # the stage alone (both frames, batch of 2), captured as its own CUDA graph and replayed between L2
                # flushes: the kernels run back to back exactly as inside the step's graph
                from vps_b200.layers import empty_nhwc
                xr = empty_nhwc(2, H, W, 3, det.act_dtype, dev)
                xr.normal_()
                det.extract_feat(xr)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    det.extract_feat(xr)
                reps = []
                for i in range(5):
                    flush.fill_(i)
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record(); g.replay(); b.record()
                    reps.append((a, b))
                torch.cuda.synchronize()
                r50_ms = sorted(a.elapsed_time(b) for a, b in reps)[len(reps) // 2]
                t = r50_ms * 1e-3
                ach = GFLOP_R50FPN_PAIR * (H * W) / float(H_FULL * W_FULL) * 1e9 / t / 1e12
                line["r50fpn_roofline"] = {"achieved": ach, "peak": peaks()["tf_sus"], "unit": "TFLOP/s",
                                           "frac": ach / peaks()["tf_sus"], "ms": r50_ms, "eager_instrumented_ms": scopes["r50fpn"][0],
                                           "note": "stage captured as its own CUDA graph, median of 5 replays with L2 flush; algorithmic 1158.4 GFLOP/pair"}
        if fast is not None:
            line["fast_mode"] = fast
        if cpu_leg is not None:
            line["cpu_baseline"] = cpu_leg
        if world == 1 and not args.no_stock:
            try:
                line["stock_pytorch_r50fpn"] = stock_pytorch_r50fpn(dev, H, W, flush)
            except Exception as ex:          # context only: never fail the bench on it
                line["stock_pytorch_r50fpn"] = {"unavailable": repr(ex)[:200]}
        print(json.dumps(line))
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    P.barrier()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="tc32", choices=["tc32", "bf16", "fp32"])
    ap.add_argument("--height", type=int, default=H_FULL)
    ap.add_argument("--width", type=int, default=W_FULL)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fast-mode", action="store_true", help="skip the bf16 fast-mode leg")
    ap.add_argument("--no-stock", action="store_true", help="skip the stock-PyTorch (cuDNN) ResNet-50-FPN context leg")
    ap.add_argument("--workload", default="pairs", choices=["pairs", "viper"],
                    help="pairs = BASELINE config 2 (1024x2048 pairs); viper = config 4 (30-frame 1088x1920 clips, one per GPU)")
    ap.add_argument("--allow-short-warmup", action="store_true", help="profiling runs under ncu only (numbers are not bench values)")
    ap.add_argument("--profile-out", default="", help="write per-call device timings of one instrumented step (JSON lines)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the results of the last step of the headline timed region (rank 0) as DIR/<name>.npy "
                         "(float32 / float64; label maps whole, seeded samples of the FPN features): the inputs are "
                         "seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if (args.impl == "b200" and not args.allow_short_warmup) else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
