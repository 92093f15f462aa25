#!/usr/bin/env python
"""Benchmark of the detection hot path (BASELINE.json metric: images/sec).

Workload at every N: SSD300 VGG-16 fp16 inference, per-GPU batch 64 of 300x300
synthetic VOC-shaped images (BASELINE.json configs[1]) -- backbone + heads
(tcgen05 convs) + anchors + decode + per-class NMS; weak scaling (images shard
batch-parallel, one NCCL all-gather of the detection records per step).

  python bench.py --gpus N --steps K --warmup W          # this framework
  python bench.py ... --dump-outputs DIR                 # + the last timed step's detections as DIR/*.npy
  python bench.py --impl reference --gpus N ...          # the reference's CPU path
                                                         # (oracle port: TF1.13 cannot run here)
One JSON line on stdout (rank 0).
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "object-detection-tensorflow_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

BATCH = 64
SIZE = 300
CFG = {"mode": "test", "data_format": "channels_last", "num_classes": 20, "weight_decay": 1e-4,
       "keep_prob": 0.5, "batch_size": BATCH, "nms_score_threshold": 0.5, "nms_max_boxes": 20,
       "nms_iou_threshold": 0.5, "pretraining_weight": None, "precision": "fp16"}
WORKLOAD = "SSD300 VGG-16 fp16 inference, batch 64/GPU, 300x300 synthetic VOC (BASELINE configs[1])"
CONV_GFLOP_PER_IMG = 62.773  # SURVEY.md App. B, real (unpadded) channels
# second workload of BASELINE.json's metric ("SSD300 & RetinaNet"): configs[2], RetinaNet FPN fp16, batch 16, 800x800
# (reference driver defaults testretinanet.py:17-41: bottleneck [3,4,6,3], 16 stem filters, max 10 boxes, IoU 0.45)
RETINA_BATCH = 16
RETINA_CFG = {"mode": "test", "data_format": "channels_last", "num_classes": 20, "weight_decay": 1e-4,
              "keep_prob": 0.5, "batch_size": RETINA_BATCH, "data_shape": [800, 800, 3], "is_bottleneck": True,
              "residual_block_list": [3, 4, 6, 3], "init_conv_filters": 16, "is_pretraining": False,
              "gamma": 2.0, "alpha": 0.25, "nms_score_threshold": 0.8, "nms_max_boxes": 10,
              "nms_iou_threshold": 0.45, "pretraining_weight": None, "precision": "fp16"}
RETINA_WORKLOAD = "RetinaNet FPN fp16 inference, batch 16/GPU, 800x800 synthetic (BASELINE configs[2]), dense-threshold NMS"
DENSE_FRACTION = 0.02  # candidates per class = 2 % of N (SURVEY 8d asks for the 1-5 % regime)


def bench_config(world):
    """`config` of the JSON line -- the same dict in both arms (ours and --impl reference)."""
    return {"workload": WORKLOAD, "global_batch": BATCH * world, "per_gpu_batch": BATCH,
            "parallelism": "dp%d (image shards, 1 all-gather of detections)" % world,
            "l2": "per-step activation working set ~2 GB >> 126 MB L2 (no reuse between steps)",
            "cuda_graph": True, "conv_gflop_per_img": CONV_GFLOP_PER_IMG,
            "pipeline": ("decode + NMS (+ all-gather) of step i run on a second stream under the first convolutions of step i+1; "
                         "candidate rows / lists / records double-buffered" if os.environ.get("ODT_PIPELINE", "1") != "0"
                         else "off: one graph per step")}


def synthetic_images(b, seed=0):
    return np.random.default_rng(seed).integers(0, 256, (b, SIZE, SIZE, 3)).astype(np.float32)


def measured_peaks():
    f = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(f):
        d = json.load(open(f))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self._kill)  # an exception inside a timed leg must not leave nvidia-smi running
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def _kill(self):
        if self.proc.poll() is None:
            self.proc.kill()
            self.proc.wait()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


_CPU_STATE = {}


def cpu_oracle_images_per_sec(n_images, repeats=1, threads=None):
    """The reference's CPU path as restated by the oracle (torch-CPU fp32 + C NMS):
    full test_one_image semantics, batch-1 graph semantics looped over images.
    The thread count is the fastest of {all cores, 64, 32, 16, 8} on this host
    (more threads than the 300x300 batch-1 convs can use only adds contention)."""
    import torch
    from odt_b200.engine import init_weights
    import SSD300
    from oracle import nets as ON
    from oracle import tails as OT
    OT.build_nms_lib()
    if "w" not in _CPU_STATE:
        model = SSD300.SSD300(dict(CFG), None)
        _CPU_STATE["w"] = init_weights(model.variables(), seed=1)
    w = _CPU_STATE["w"]
    img = synthetic_images(max(n_images, 1), seed=0)

    def one(i):
        preds = ON.ssd_heads(w, img[i:i + 1], SIZE)
        OT.ssd_detect(preds, SIZE, CFG["nms_score_threshold"], CFG["nms_max_boxes"],
                      CFG["nms_iou_threshold"])

    if threads is None and "threads" not in _CPU_STATE:
        ncpu = os.cpu_count() or 1
        best_t, best_dt = ncpu, None
        for t in sorted({ncpu, min(ncpu, 64), min(ncpu, 32), min(ncpu, 16), min(ncpu, 8)}, reverse=True):
            torch.set_num_threads(t)
            one(0)  # warm-up (thread pool, oneDNN primitive cache)
            t0 = time.perf_counter()
            one(0)
            dt = time.perf_counter() - t0
            if best_dt is None or dt < best_dt:
                best_t, best_dt = t, dt
        _CPU_STATE["threads"] = best_t
    threads = threads or _CPU_STATE["threads"]
    torch.set_num_threads(threads)
    one(0)
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        for i in range(n_images):
            one(i)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return n_images / best, threads


_OUT = None


def emit(line):
    out = _OUT if _OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path.  TF 1.13
    is not installable here and SSD300.py does not parse, so this times the oracle
    port (kind 'port') on all host cores; each step is a bounded sample of the workload."""
    if rank != 0:
        return
    sample = 4
    vals = []
    t_all = time.perf_counter()
    for _ in range(args.steps):
        v, threads = cpu_oracle_images_per_sec(sample)
        vals.append(v)
        if time.perf_counter() - t_all > 240:
            break
    v = float(np.mean(vals))
    line = {"impl": "reference", "metric": "images/sec", "value": v, "unit": "images/sec",
            "n_gpus": args.gpus, "steps": len(vals), "warmup": args.warmup,
            "ms_per_step": 1e3 * sample / v, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(args.gpus),
            "cpu_baseline": {"value": v, "unit": "images/sec", "cores": threads, "kind": "port",
                             "sample": "%d images per step, batch-1 graph semantics, torch-CPU fp32 "
                                       "convs + C NMS" % sample},
            "e2e": {"value": v, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def dense_threshold(net, fraction=DENSE_FRACTION):
    """Bench SETUP (untimed, plain torch on the rows the GPU produced): the softmax-family score threshold at
    which `fraction` * N candidates per class and image pass, so that decode compaction and NMS do real work
    with random-init weights (ADVICE r1: report candidate load; SURVEY 8d: dense regime)."""
    import torch
    rows = net.head_buf
    probs = torch.softmax(rows[..., :21], dim=-1)
    fg = probs[..., :20][probs.argmax(dim=-1) < 20]          # rows whose arg-max is not background
    want = int(fraction * net.N * 20 * net.batch)
    flat = fg.reshape(-1)
    if flat.numel() == 0:
        return None
    k = min(max(want, 1), flat.numel())
    return float(torch.topk(flat, k, sorted=True).values[-1].item()) if k < 50_000_000 else float(flat.min().item())


def timed_ops(net, pick, reps=5):
    """Eager per-launch CUDA-event timing inside whole forwards (realistic cache state), called straight after the
    timed resident leg so that the clocks are in the same sustained state: returns the MEDIAN over `reps` forwards (after
    two untimed ones) of the per-forward milliseconds of the ops `pick(op)` selects, of the decode launch and of the
    NMS launch."""
    import torch
    st = torch.cuda.current_stream().cuda_stream
    t = net.tail
    per_fwd, dec, nms = [], [], []
    torch.cuda.synchronize()

    def ev():
        return torch.cuda.Event(enable_timing=True)

    for rep in range(reps + 2):
        evs = []
        if getattr(net, "gn_arena", None) is not None:
            net.gn_arena.zero_()
        for op in net.ops:
            if pick(op):
                a, b = ev(), ev()
                a.record()
                op.launch(net, st)
                b.record()
                evs.append((a, b))
            else:
                op.launch(net, st)
        e = [ev() for _ in range(3)]
        e[0].record()
        t.launch_decode(net, st)
        e[1].record()
        t.launch_nms(net, st)
        e[2].record()
        if rep >= 2:
            per_fwd.append(evs)
            dec.append((e[0], e[1]))
            nms.append((e[1], e[2]))
    torch.cuda.synchronize()
    med = lambda xs: sorted(xs)[len(xs) // 2]
    return (med([sum(a.elapsed_time(b) for a, b in evs) for evs in per_fwd]),
            med([a.elapsed_time(b) for a, b in dec]), med([a.elapsed_time(b) for a, b in nms]))


def dump_detections(out_dir, name, tail):
    """What a caller of the timed step receives: the Detections of the step's packed records (scores [B,D],
    boxes [B,D,4] as y1,x1,y2,x2, class ids [B,D], counts [B]), slots past each image's count zeroed, written as
    float32 to out_dir/<name>_<array>.npy.  Inputs and weights are seeded, so two builds can be compared file by file."""
    from odt_b200.engine import unpack_records
    det = unpack_records(tail.rec.cpu().numpy(), tail.p.cap)
    valid = np.arange(det.scores.shape[1])[None, :] < det.count[:, None]
    arrays = {"scores": np.where(valid, det.scores, 0), "boxes": np.where(valid[..., None], det.boxes, 0),
              "class_id": np.where(valid, det.class_id, 0), "count": det.count}
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, "%s_%s.npy" % (name, k)), np.asarray(v, np.float32))


def tail_launch_floor_us():
    """The same two tail launches (memset + decode, memsets + NMS) on a 32-row input: the launch-bound floor."""
    import numpy as np
    import torch
    from odt_b200 import nets
    from odt_b200.engine import RowsHarness
    cfg = dict(CFG)
    rows = np.zeros((1, 38 * 38 * 4, 25), np.float32)
    h = RowsHarness(nets.ssd_tail(300, cfg), [(38, 38, 4)], rows)
    st = torch.cuda.current_stream().cuda_stream
    for _ in range(3):
        h.tail.launch(h, st)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(20):
        h.tail.launch(h, st)
    b.record()
    torch.cuda.synchronize()
    return 1e3 * a.elapsed_time(b) / 20


def tail_roofline(net, dec_ms, nms_ms, peaks, floor_us):
    t = net.tail
    rd = net.head_buf.numel() * 4                      # N*25*4 B per image (SURVEY 8d)
    wr = net.batch * t.D * 24                          # D_max*24 B per image
    us = 1e3 * (dec_ms + nms_ms)
    gbs = (rd + wr) / (us * 1e-6) / 1e9
    cc = t.cand_count.cpu().numpy()
    return {"bytes_per_step": int(rd + wr), "decode_us": 1e3 * dec_ms, "nms_us": 1e3 * nms_ms, "gbs": gbs,
            "decode_gbs": rd / (dec_ms * 1e-3) / 1e9,
            "frac_of_hbm": gbs / float(peaks["hbm_gbs"]), "decode_frac_of_hbm": rd / (dec_ms * 1e-3) / 1e9 / float(peaks["hbm_gbs"]),
            "hbm_peak_gbs": float(peaks["hbm_gbs"]), "launch_floor_us": floor_us,
            "score_threshold": float(t.p.score_thr),
            "candidates_per_class_mean": float(cc.mean()), "candidates_per_class_max": int(cc.max()),
            "dets_per_image_mean": float(t.det_count.float().mean().item()),
            "timing": "CUDA events around the two launches inside eager whole forwards (rows just written by the head "
                      "convs, i.e. the cache state of the real step), mean of 3"}


def conv_roofline(net, tc_ms, ms_step, peaks, peak_src, kname):
    from odt_b200.engine import ConvOp
    tc_ops = [op for op in net.ops if isinstance(op, ConvOp) and getattr(op, "use_tc", False)]
    tc_flops = sum(op.flops for op in tc_ops)
    sus = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
    burst = float(peaks.get("bf16_tflops", sus))
    achieved = tc_flops / (tc_ms * 1e-3) / 1e12
    whole = net.conv_flops / (ms_step * 1e-3) / 1e12
    return {"bound": "tensor", "kernel": kname, "achieved": achieved, "peak": sus, "unit": "TFLOP/s",
            "frac": achieved / sus, "frac_sustained": achieved / sus, "frac_burst": achieved / burst,
            "peak_burst": burst,
            "peak_source": peak_src + " cuBLAS bf16: `peak`/`frac` use the sustained figure (the kernels are timed inside "
                                      "back-to-back whole steps), frac_burst the best-of-10 burst figure",
            "launches_per_step": len(tc_ops), "tc_ms_per_step": tc_ms,
            "algorithmic_gflop_per_step": tc_flops / 1e9, "share_of_step": tc_ms / ms_step,
            "timing": "CUDA events around every launch of these kernels inside eager whole forwards straight after the timed "
                      "resident leg (same sustained clock state), median of 5 forwards",
            "whole_step_tflops": whole, "whole_step_frac_sustained": whole / sus, "whole_step_frac_burst": whole / burst}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-retinanet", action="store_true", help="skip the second workload (RetinaNet-800 B=16)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the detections of each workload's last timed step to DIR/*.npy")
    args = ap.parse_args()
    assert args.warmup >= 0 and args.steps >= 1

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries exactly ONE JSON line: keep the real stdout aside and point fd 1 at stderr so
    # that libraries writing to stdout (NCCL's version banner, ...) cannot pollute it
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the one JSON line
    import torch
    import torch.distributed as tdist
    from odt_b200 import dist as od
    import __graft_entry__ as ge
    rank, world, local = od.init_from_env()
    if not os.path.exists(os.path.join(ROOT, "object-detection-tensorflow_b200", "odt_b200",
                                       "libodt_b200.so")):
        if rank == 0:
            ge.build()
        if world > 1:
            tdist.barrier()
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d" % args.gpus
    W = max(args.warmup, 3)
    K = args.steps
    peaks, peak_src = measured_peaks()

    def barrier():
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        return float(t.item())

    def time_resident(net, gathered, sampler=None):
        """W warm-up + K timed device-resident steps (graph replay + the records' all-gather at N > 1).  Default: the
        two-stage pipeline of the engine (decode + NMS + gather of step i on a second stream under the first
        convolutions of step i+1, everything the tail touches double-buffered); ODT_PIPELINE=0: one graph per step.
        Returns (ms of the K steps, the Tail holding the last step's records)."""
        pipelined = os.environ.get("ODT_PIPELINE", "1") != "0"
        if pipelined:
            net.capture_pipelined()
        counter = [0]
        last = [net.tail]

        def step():
            if pipelined:
                last[0] = net.run_pipelined(counter[0] & 1,
                                            (lambda t: od.gather_records(t.rec, out=gathered)) if world > 1 else None)
                counter[0] += 1
                return
            net.run()
            if world > 1:
                od.gather_records(net.tail.rec, out=gathered)
        for _ in range(W):
            step()
        if sampler is not None:
            t_spin = time.perf_counter()
            again = torch.tensor([1], device="cuda")
            while True:  # keep the GPU under the same load until nvidia-smi has sampled once (all ranks agree)
                again[0] = 1 if (len(sampler.lines) < 1 and time.perf_counter() - t_spin < 3.0) else 0
                if world > 1:
                    tdist.all_reduce(again, op=tdist.ReduceOp.MAX)
                if int(again.item()) == 0:
                    break
                for _ in range(4):
                    step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            step()
        if pipelined:
            net.join_pipelined()  # the closing event waits for the last tails as well
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)), last[0]

    def time_e2e(model, images, sampler=None):
        """Public API, host buffers: pinned H2D of every step's images + D2H of every step's records inside
        the timed region (detect_stream; sharded with rank 0 as the consumer of the gathered records).  Like the
        resident leg, the warm-up keeps the GPU under this same load until nvidia-smi has sampled once, so both
        legs are timed in the sustained (power-capped) clock state rather than one of them in a cool burst."""
        def run(n):
            for res in model.detect_stream((images for _ in range(n)), sharded=world > 1, consumer=0):
                assert len(res) in (images.shape[0], images.shape[0] * world)
        run(W)
        if sampler is not None:
            t_spin = time.perf_counter()
            again = torch.tensor([1], device="cuda")
            while True:
                again[0] = 1 if (len(sampler.lines) < 1 and time.perf_counter() - t_spin < 3.0) else 0
                if world > 1:
                    tdist.all_reduce(again, op=tdist.ReduceOp.MAX)  # all ranks leave the (collective) loop together
                if int(again.item()) == 0:
                    break
                run(4)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(K)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    def e2e_bytes(net, images):
        # whole job, per step: every rank uploads its shard and reads back its own records; at N > 1 the
        # consumer rank reads back the gathered records of all N shards instead
        rec = net.tail.rec.numel() * 4
        return int(images.numel() * 4) * world, int(rec if world == 1 else rec * world + rec * (world - 1))

    # ======================= workload 1 (headline): SSD300 B=64 ====================================
    import SSD300
    model = SSD300.SSD300(dict(CFG), None)
    net = model.engine(BATCH)  # builds, uploads seeded weights (identical on every rank), captures the graph
    images = torch.from_numpy(synthetic_images(BATCH, seed=rank)).pin_memory()
    net.image_buf.copy_(images)
    gathered = (torch.empty((world * BATCH, net.tail.rec.shape[1]), dtype=torch.float32, device="cuda")
                if world > 1 else None)
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()  # started before the warm-up so that samples exist for short timed regions
    ms_total, last_tail = time_resident(net, gathered, sampler)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_detections(args.dump_outputs, "ssd300", last_tail)
    ms_step = ms_total / K
    value = world * BATCH * K / (ms_total / 1e3)
    from odt_b200.engine import ConvOp
    is_tc = lambda op: isinstance(op, ConvOp) and getattr(op, "use_tc", False)
    tc_ms, dec_ms, nms_ms = timed_ops(net, is_tc)  # straight after the resident leg: same clock state
    sampler2 = ClockSampler(local)
    sampler2.start()
    ms_e2e = time_e2e(model, images, sampler2)
    e2e_clocks = sampler2.stop()
    e2e_value = world * BATCH * K / (ms_e2e / 1e3)
    h2d, d2h = e2e_bytes(net, images)

    roofline = conv_roofline(net, tc_ms, ms_step, peaks, peak_src,
                             "tcgen05 implicit-GEMM convolutions (conv_tc_kernel<1|2>, conv_tapn_kernel where planned)")
    traffic, traffic_src = None, None
    for cand in ("r02_conv_traffic.json", "r01_conv_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", cand)
        if os.path.exists(tpath):  # committed ncu measurement of the same command (scripts/conv_traffic.py)
            with open(tpath) as f:
                tj = json.load(f)
            if tj.get("launches_per_step") == roofline["launches_per_step"]:
                traffic, traffic_src = tj["dram_bytes_per_launch_avg"], "profiles/%s (ncu dram__bytes_read+write)" % cand
                break
    roofline["traffic"], roofline["traffic_source"] = traffic, traffic_src
    floor_us = tail_launch_floor_us()
    ssd_tail_rf = tail_roofline(net, dec_ms, nms_ms, peaks, floor_us)

    cfg_line = bench_config(world)
    cfg_line["conv_roofline_frac_whole_step"] = roofline["whole_step_frac_sustained"]
    line = {"metric": "images/sec", "value": value, "unit": "images/sec", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": cfg_line,
            "e2e": {"value": e2e_value, "unit": "images/sec", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / K, "clocks": e2e_clocks,
                    "mode": "detect_stream (two-stage pipeline, read-back one step behind)" if world == 1 else
                            "detect_stream sharded, consumer rank 0 reads the all-gathered records"},
            "gpu_launches": net.num_launches() * K,
            "roofline": roofline, "clocks": clocks,
            "tail_roofline_ssd300": ssd_tail_rf}

    # ======================= workload 2: RetinaNet-800 B=16, dense-threshold NMS =====================
    if not args.no_retinanet:
        del gathered
        model._engines.clear()
        del net, model
        torch.cuda.empty_cache()
        import RetinaNet
        rmodel = RetinaNet.RetinaNet(dict(RETINA_CFG), None)
        rnet = rmodel.engine(RETINA_BATCH, graph=False)
        rimg = torch.from_numpy(np.random.default_rng(100 + rank).integers(
            0, 256, (RETINA_BATCH, 800, 800, 3)).astype(np.float32)).pin_memory()
        rnet.image_buf.copy_(rimg)
        rnet.forward()
        torch.cuda.synchronize()
        thr = dense_threshold(rnet)
        if world > 1:  # one threshold for the job: rank 0's
            tt = torch.tensor([thr if thr is not None else -1.0], dtype=torch.float64, device="cuda")
            tdist.broadcast(tt, 0)
            thr = float(tt.item()) if tt.item() >= 0 else None
        if thr is not None:
            # the Tail's own attribute too: capture_pipelined() prepares the second pipeline slot's tail from it
            rnet.tail.score_thr = rnet.tail.p.score_thr = thr
            rmodel.nms_score_threshold = thr
        rnet.capture()
        rg = (torch.empty((world * RETINA_BATCH, rnet.tail.rec.shape[1]), dtype=torch.float32, device="cuda")
              if world > 1 else None)
        rs1 = ClockSampler(local)
        rs1.start()
        r_ms_total, r_last_tail = time_resident(rnet, rg, rs1)
        r_clocks = rs1.stop()
        if args.dump_outputs and rank == 0:
            dump_detections(args.dump_outputs, "retinanet800", r_last_tail)
        r_ms_step = r_ms_total / K
        r_tc_ms, r_dec_ms, r_nms_ms = timed_ops(rnet, is_tc)
        rs2 = ClockSampler(local)
        rs2.start()
        r_e2e_ms = time_e2e(rmodel, rimg, rs2)
        r_e2e_clocks = rs2.stop()
        rh2d, rd2h = e2e_bytes(rnet, rimg)
        rr = conv_roofline(rnet, r_tc_ms, r_ms_step, peaks, peak_src, "tcgen05 implicit-GEMM convolutions")
        rr["note"] = ("tc_ms_per_step is the SERIALISED sum of the kernels' eager durations; the graph runs the FPN levels and the "
                      "two towers on parallel lanes, so share_of_step can exceed 1 and whole_step_frac_* is the figure for the step")
        line["workloads"] = {"retinanet800_b16": {
            "workload": RETINA_WORKLOAD, "value": world * RETINA_BATCH * K / (r_ms_total / 1e3), "unit": "images/sec",
            "ms_per_step": r_ms_step, "per_gpu_batch": RETINA_BATCH, "gpu_launches": rnet.num_launches() * K,
            "clocks": r_clocks,
            "e2e": {"value": world * RETINA_BATCH * K / (r_e2e_ms / 1e3), "unit": "images/sec",
                    "ms_per_step": r_e2e_ms / K, "h2d_bytes_per_step": rh2d, "d2h_bytes_per_step": rd2h,
                    "clocks": r_e2e_clocks},
            "roofline": rr}}
        line["tail_roofline"] = tail_roofline(rnet, r_dec_ms, r_nms_ms, peaks, floor_us)
        line["tail_roofline"]["workload"] = "retinanet800_b16"

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, threads = cpu_oracle_images_per_sec(64)
        line["cpu_baseline"] = {"value": v, "unit": "images/sec", "cores": threads, "kind": "port",
                                "sample": "one whole batch (64 images, ~5-10 s), oracle port (torch-CPU fp32 + C NMS), "
                                          "batch-1 graph semantics like the reference"}
    if rank == 0:
        emit(line)
    if world > 1:
        tdist.barrier()
        tdist.destroy_process_group()


if __name__ == "__main__":
    main()
