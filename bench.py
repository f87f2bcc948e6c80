#!/usr/bin/env python
"""Region-stage benchmark (BASELINE.json metric: region-stage images/sec; NMS us @12k boxes).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload all|rpn|voc1|train|infer|joint]
                    [--dump-outputs DIR]

The line's headline (`value`, `e2e`, `roofline`, `cpu_baseline`) is BASELINE.json configs[1]: RPN proposal layer, 9 anchors x
38x63 map (608x1008 image, N = 21546), 12000 pre-NMS -> 2000 post-NMS at IoU 0.7, batch 64 images per GPU; one "step" = one
pass of decode + top-k + NMS over one batch of 64 synthetic images.  With the default `--workload all` the same line carries
`sub_results` for the other single-GPU configurations of the metric, measured by the same process under the same clock:
    voc1  = configs[0]: one 600x1000 VOC image, FRCNN.predict's region path (6000 -> 300, RoIPool 300, D1, 21-class NMS), latency
    train = configs[2]: target makers + RoIPool 7x7 fwd/bwd, 16 images/GPU
    infer = configs[3]: COCO-shaped 800x1333 inference, 81 classes, 8 images/GPU, detections all-gathered over NCCL
Under torchrun every rank processes its own images (weak scaling; the only collective is the detection all-gather of
`infer`); rank 0 prints ONE JSON line.  `--impl reference` times the CPU restatement of the reference (oracle/) on the
host cores for the same configurations.

`--steps K` is the number of timed steps of every workload's step loops (the per-kernel timings use their own repetition
counts).  `--dump-outputs DIR` writes, after the timed steps, what the timed path of each workload run handed its caller in
its last step as DIR/<workload>_<output>.npy (float32, or float64 for integer outputs); inputs are seeded, so two builds
run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

HW = (608, 1008)
BATCH = 64
PRE_K, POST_K, THR = 12000, 2000, 0.7
N_ROTATE = 8           # resident input batches cycled through so that every step reads cold data (> L2)
DUMP_SAMPLE = 1 << 20  # --dump-outputs: an output with more elements is reduced to this many seeded positions
DUMP_MAX_BYTES = 64 << 20
METRIC = "region-stage images/sec (RPN+NMS+RoIPool) at 1/2/4/8 B200; NMS us @12k boxes"
WORKLOAD = ("configs[1]: RPN proposal layer, 9 anchors x 38x63 map (608x1008), 12000 pre-NMS -> 2000 post-NMS "
            "@ IoU 0.7, batch 64 images/GPU")
W_VOC1 = ("configs[0]: VOC VGG16 inference region path, 1 image 600x1000: proposals 6000 -> 300 @0.7, RoIPool 300 x 512 x 7x7, "
          "per-class decode, 21-class NMS @0.3 (thres 0.05)")
W_TRAIN = ("configs[2]: training targets (256 anchor / 128 RoI sampling, G=8) + RoIPool 7x7 fwd/bwd on 512-ch stride-16 "
           "features (37x62), batch 16 images/GPU, RoIs sampled from the RPN proposals")
W_INFER = ("configs[3]: COCO-shaped 800x1333 inference, 81 classes, 6000 -> 300 proposals, RoIPool of 300 RoIs x 512 ch, "
           "80-class NMS @0.3 (thres 0.05), 8 images/GPU, detections [8,100,6] all-gathered")


def config_of(workload: str, batch: int) -> dict:
    """Identical in both arms (`--impl ours` / `--impl reference`)."""
    return {"workload": workload, "images_per_gpu_per_step": batch,
            "l2": "GPU arm: every step reads a different resident input set and the rotation is larger than the 126 MB L2 "
                  "(sizes in config_detail); CPU reference arm: not applicable"}


def profile_counters(kernel: str) -> dict:
    """Per-launch counters of `kernel` from the committed ncu --set full capture (profiles/traffic.json)."""
    try:
        return json.load(open(os.path.join(REPO, "profiles", "traffic.json")))[kernel]
    except (OSError, KeyError, ValueError):
        return {}


def ncu_traffic(kernel: str):
    t = profile_counters(kernel)
    try:
        return t["dram_bytes_read"] + t["dram_bytes_write"]
    except KeyError:
        return None


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
            return float(d["hbm_gbs"]), "measured", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback", 1965.0


def make_inputs(seed0: int, batch: int, hw=HW):
    from faster_rcnn_pytorch_b200 import synth
    n = synth.num_anchors(hw)
    rs = np.random.RandomState(seed0)
    logits = rs.standard_normal((batch, n, 2)).astype(np.float32)
    reg = (rs.standard_normal((batch, n, 4)) * 0.2).astype(np.float32)
    return logits, reg


def dump_arrays(prefix: str, arrays: dict) -> dict:
    """Host copies of one step's outputs for --dump-outputs: floating-point outputs as float32 (float64 stays float64),
    integer ones as float64 (exact).  An output of more than DUMP_SAMPLE elements is reduced to its elements at seeded
    positions of the flattened array (name suffix `_sample`), the same positions in every run."""
    import torch
    out = {}
    for key, t in arrays.items():
        t = torch.as_tensor(t).detach()
        name = f"{prefix}_{key}"
        if t.numel() > DUMP_SAMPLE:
            pos = np.unique(np.random.RandomState(0).randint(0, t.numel(), DUMP_SAMPLE))
            t = t.reshape(-1)[torch.from_numpy(pos).to(t.device)]
            name += "_sample"
        wide = t.dtype == torch.float64 or not t.is_floating_point()
        out[name] = t.to(torch.float64 if wide else torch.float32).cpu().numpy()
    return out


def write_outputs(dumps: dict, out_dir: str):
    total = sum(a.nbytes for a in dumps.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs: {total / 2**20:.1f} MB of outputs, more than {DUMP_MAX_BYTES >> 20} MB")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in dumps.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------ CPU arm (oracle port)
def _cpu_pool(fn, n_images: int, threads: int):
    """Images are independent (the reference is batch-1): one image per worker thread; numpy and the C helpers of the
    oracle release the GIL."""
    from concurrent.futures import ThreadPoolExecutor
    fn(0)  # warm-up
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(fn, range(n_images)))
    dt = time.perf_counter() - t0
    return n_images / dt, dt


def cpu_rpn(n_images: int, threads: int, seed0: int = 2000):
    """configs[1] on the host: RegionProposal.forward (models/model.py:17-58) per image."""
    from oracle import region_oracle as orc, _cbridge
    _cbridge.load(required=True)
    from faster_rcnn_pytorch_b200 import synth
    anchor = orc.enumerate_anchors(HW)
    ins = [synth.rpn_head_outputs(seed0 + i, HW)[:2] for i in range(n_images)]
    return _cpu_pool(lambda i: orc.region_proposal(ins[i][0], ins[i][1], anchor, "train")["rois"].shape[0], n_images, threads)


def cpu_predict(n_images: int, threads: int, hw, num_classes: int, seed0: int):
    """configs[0] / configs[3] on the host: FRCNN.predict's region path (models/model.py:346-402) per image: proposal layer
    in test mode, RoIPool of the 300 rois, per-class decode, per-class NMS."""
    from oracle import region_oracle as orc, _cbridge
    _cbridge.load(required=True)
    from faster_rcnn_pytorch_b200 import synth
    anchor = orc.enumerate_anchors(hw)
    fh, fw = hw[0] // 16, hw[1] // 16
    rs = np.random.RandomState(seed0)
    feat = rs.standard_normal((1, 512, fh, fw)).astype(np.float32)
    ins = [synth.rpn_head_outputs(seed0 + i, hw)[:2] for i in range(n_images)]
    heads = [synth.head_outputs(seed0 + 50 + i, 300, num_classes) for i in range(n_images)]

    def one(i):
        rois = orc.region_proposal(ins[i][0], ins[i][1], anchor, "test")["rois"]
        pooled, _ = orc.roi_pool_forward(feat, orc.scale_rois(rois, fh, fw))
        r = rois.shape[0]
        prob, boxes = orc.decode_classwise(heads[i][0][:r], heads[i][1][:r], rois, num_classes)
        return orc.suppress(boxes, prob, num_classes, 0.05)[0].shape[0] + int(pooled.shape[0])

    return _cpu_pool(one, n_images, threads)


def cpu_train(n_images: int, threads: int, seed0: int = 3000):
    """configs[2] on the host: RPNTargetMaker + FastRcnnTargetMaker (models/model.py:123-266) + RoIPool 7x7 forward and
    backward of the 128 sampled rois, per image (proposals precomputed, as on the GPU arm)."""
    from oracle import region_oracle as orc, _cbridge
    _cbridge.load(required=True)
    from faster_rcnn_pytorch_b200 import synth
    hw = (600, 1000)
    fh, fw = hw[0] // 16, hw[1] // 16
    anchor = orc.enumerate_anchors(hw)
    rs = np.random.RandomState(seed0)
    feat = rs.standard_normal((1, 512, fh, fw)).astype(np.float32)
    gout = rs.standard_normal((128, 512, 7, 7)).astype(np.float32)
    props = [synth.random_boxes(seed0 + 100 + i, 2000)[0] for i in range(n_images)]
    gts = [synth.gt_boxes(seed0 + i, 8) for i in range(n_images)]

    def one(i):
        rp = orc.HostRandperm(seed0 + i)
        orc.rpn_targets(gts[i][0], anchor, rp)
        f = orc.frcnn_targets(gts[i][0], gts[i][1], props[i], rp)
        rois5 = orc.scale_rois(f["sample_rois"], fh, fw)
        out, arg = orc.roi_pool_forward(feat, rois5)
        gin = orc.roi_pool_backward(gout[:rois5.shape[0]], arg, rois5, feat.shape)
        return float(gin[0, 0, 0, 0])

    return _cpu_pool(one, n_images, threads)


CPU_ARMS = {
    "rpn": (lambda n, t: cpu_rpn(n, t), WORKLOAD, BATCH, "numpy decode/sort + C NMS"),
    "voc1": (lambda n, t: cpu_predict(n, t, (600, 1000), 21, 1000), W_VOC1, 1, "numpy decode/sort + C NMS + C RoIPool + numpy per-class decode / NMS loop"),
    "train": (lambda n, t: cpu_train(n, t), W_TRAIN, 16, "numpy target makers (mt19937 randperm replay) + C RoIPool fwd/bwd"),
    "infer": (lambda n, t: cpu_predict(n, t, (800, 1333), 81, 4000), W_INFER, 8, "numpy decode/sort + C NMS + C RoIPool + numpy per-class decode / NMS loop"),
}


def torchvision_cpu_nms_ms(n: int = 12000, post: int = 2000):
    """BASELINE.md section 3: the reference's own NMS call (torchvision.ops.nms on CPU tensors, models/model.py:53) on
    one image's score-sorted RPN boxes, beside the oracle port's C kernel on the same boxes.  (ms, ms) or None."""
    try:
        import torch
        import torchvision
        from oracle import region_oracle as orc, _cbridge
        _cbridge.load(required=True)
        from faster_rcnn_pytorch_b200 import synth
        _, reg, scores = synth.rpn_head_outputs(2000, HW)
        boxes = orc.decode_clip(reg, orc.enumerate_anchors(HW))
        valid = orc.min_size_mask(boxes)
        order = orc.sort_desc(scores[valid])[:n]
        tb = np.ascontiguousarray(boxes[valid][order])
        sc = np.arange(len(tb), 0, -1).astype(np.float32)
        tt, ts = torch.from_numpy(tb), torch.from_numpy(sc)
        torchvision.ops.nms(tt, ts, 0.7)
        t0 = time.perf_counter(); k_tv = torchvision.ops.nms(tt, ts, 0.7)[:post]; t_tv = time.perf_counter() - t0
        t0 = time.perf_counter(); k_or = orc.nms(tb, sc, 0.7)[:post]; t_or = time.perf_counter() - t0
        same = bool(np.array_equal(k_tv.numpy(), k_or))
        return {"torchvision_cpu_nms_ms": 1e3 * t_tv, "oracle_c_nms_ms": 1e3 * t_or, "keep_lists_equal": same,
                "what": f"one image, {len(tb)} score-sorted RPN boxes -> first {post} keeps @0.7, single call"}
    except Exception as e:  # torchvision missing on the box: the port alone stands
        return {"unavailable": str(e)[:120]}


def cpu_baseline(name: str, threads: int, per_thread: int = 2) -> dict:
    fn, _, _, how = CPU_ARMS[name]
    sample = max(threads, 8) * per_thread
    v, dt = fn(sample, threads)
    out = {"value": v, "unit": "images/s", "cores": threads, "kind": "port",
           "sample": f"{sample} images of the same workload, oracle port ({how}), one image per thread on {threads} "
                     f"threads, {dt:.1f} s wall"}
    if name == "rpn":
        out["nms_kernel_check"] = torchvision_cpu_nms_ms()
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    sample = max(threads, 8) * 4
    for _ in range(args.warmup):
        cpu_rpn(min(sample, threads), threads)
    t_tot = 0.0
    for _ in range(args.steps):
        _, dt = cpu_rpn(sample, threads)
        t_tot += dt
    value = sample * args.steps / t_tot
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(WORKLOAD, BATCH),
        "cpu_baseline": {"value": value, "unit": "images/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} images/step of the same workload, oracle port (numpy decode/sort + C NMS), "
                                   f"one image per thread on {threads} threads"},
        "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if args.workload == "all":
        sub = {}
        for name in ("voc1", "train", "infer"):
            cb = cpu_baseline(name, threads)
            _, wl, batch, _ = CPU_ARMS[name]
            sub[name] = {"value": cb["value"], "unit": "images/s", "config": config_of(wl, batch), "cpu_baseline": cb,
                         "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        line["sub_results"] = sub
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ GPU arm
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "50"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
            atexit.register(self.stop)        # a run that fails must not leave nvidia-smi behind
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        p, self.p = self.p, None
        p.terminate()
        try:
            p.wait(timeout=5)
        except Exception:
            p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.f.read().splitlines():
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for nm, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if sm:
            hi = [s for s in sm if s >= 0.5 * max(sm)]   # samples under load
            out = {"sm_mhz": float(np.median(hi)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


class Ctx:
    """Process-wide plumbing of the GPU arm: device, NCCL group, device-side timing (max over ranks)."""

    def __init__(self, dump: bool = False):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (the region stage has no CPU path; use --impl reference)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        # pinned staging buffers are allocated (first touch) by this thread: keep it on the GPU's NUMA node
        from faster_rcnn_pytorch_b200 import hostpin
        self.numa = hostpin.bind_host_thread_to_gpu_node(self.local) if self.world > 1 else {"bound": False}
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        from faster_rcnn_pytorch_b200 import _lib
        self._lib = _lib
        self.lib = _lib.load()
        self.peak, self.peak_how, self.sm_mhz = peaks()
        self.num_sms = int(torch.cuda.get_device_properties(self.dev).multi_processor_count)
        self.dump = dump and self.rank == 0
        self.dumps = {}

    def keep_outputs(self, prefix: str, arrays: dict):
        """--dump-outputs: keep host copies of what the timed path's last step handed its caller (rank 0)."""
        if self.dump:
            self.dumps.update(dump_arrays(prefix, arrays))

    def sync_all(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def maxms(self, ms: float) -> float:
        if self.world > 1:
            t = self.torch.tensor([ms], device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def timed(self, fn, steps: int, tail=None) -> float:
        """ms for `steps` calls of fn(i): barrier + synchronize on both sides, CUDA events, max over ranks."""
        torch = self.torch
        self.sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        if tail is not None:
            tail()
        e1.record()
        torch.cuda.synchronize()
        ms = self.maxms(e0.elapsed_time(e1))
        self.sync_all()
        return ms

    def median_ms(self, fn, steps: int, runs: int = 5, tail=None) -> float:
        return float(np.median([self.timed(fn, steps, tail) for _ in range(runs)]))

    def graph_of(self, fn):
        """Capture fn() (kernels + torch allocations from the graph's private pool) into a CUDA graph, or None."""
        torch = self.torch
        try:
            fn()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                out = fn()
            return g, out
        except RuntimeError:
            torch.cuda.synchronize()
            return None, None

    def kernel_ms(self, fn, reps: int) -> float:
        """Average device time of one launch of fn(i, stream): `reps` launches captured into a CUDA graph, the replay
        bracketed by events on the launching stream -- the kernel's duration plus the device-side launch gap, not the
        interval at which Python can issue ctypes calls."""
        torch = self.torch
        st = torch.cuda.current_stream().cuda_stream
        for i in range(N_ROTATE):
            fn(i, st)
        self.sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                cs = torch.cuda.current_stream().cuda_stream
                for i in range(reps):
                    fn(i, cs)
            g.replay()
            torch.cuda.synchronize()
            e0.record()
            g.replay()
            e1.record()
        except RuntimeError:
            torch.cuda.synchronize()
            e0.record()
            for i in range(reps):
                fn(i, st)
            e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def _issue_roofline(ctx, kernel: str, ms: float, sms: int = 148) -> dict:
    """Instruction-issue roofline of a latency / ALU-bound kernel: executed warp instructions per launch (ncu
    smsp__inst_executed.sum of the committed capture: same kernel, same launch geometry, same inputs, deterministic) /
    live duration, against the issue rate of the SMs the launch occupies (`sms` x 4 schedulers x SM clock: with several
    batches in flight the other SMs run the neighbouring batches' kernels)."""
    c = profile_counters(kernel)
    inst = c.get("inst_executed")
    peak = sms * 4 * ctx.sm_mhz * 1e6 / 1e9      # G warp-instructions / s
    ach = inst / (ms * 1e-3) / 1e9 if inst else None
    return {"kernel": kernel, "bound": "issue", "achieved": ach, "peak": peak, "unit": "Gwarp-inst/s",
            "frac": (ach / peak) if ach else None, "traffic": ncu_traffic(kernel),
            "inst_executed_per_launch": inst, "peak_source": f"{sms} SMs occupied x 4 schedulers x {ctx.sm_mhz:.0f} MHz",
            "note": "neither HBM- nor tensor-bound: ~0.2 MB of boxes per image; see DESIGN.md 4.3"}


def _hbm_roofline(ctx, kernel: str, nbytes: float, ms: float, **extra) -> dict:
    ach = nbytes / (ms * 1e-3) / 1e9
    d = {"kernel": kernel, "bound": "hbm", "achieved": ach, "peak": ctx.peak, "unit": "GB/s", "frac": ach / ctx.peak,
         "traffic": ncu_traffic(kernel), "peak_source": ctx.peak_how, "bytes_per_launch": nbytes}
    d.update(extra)
    return d


# ------------------------------------------------------------------------------------------ configs[1]
def verify_proposals(plan, rois, count, images) -> bool:
    """Outside every timed region: the given images of the plan's last run against the oracle fed the GPU's own decoded
    boxes / scores (index-valued stages from identical fp32 inputs)."""
    from oracle import region_oracle as orc, _cbridge
    _cbridge.load(required=True)
    it = plan.intermediates()
    rois_h, count_h = rois.cpu().numpy(), count.cpu().numpy()
    ok = True
    for i in images:
        boxes = it["boxes"][i].cpu().numpy()
        valid = it["valid"][i].cpu().numpy().astype(bool)
        sc = it["scores"][i].cpu().numpy()
        ok &= bool(np.array_equal(valid, orc.min_size_mask(boxes)))
        src = np.nonzero(valid)[0]
        order = src[orc.sort_desc(sc[valid])[:plan.pre_k]]
        n = len(order)
        ok &= int(it["top_count"][i]) == n and bool(np.array_equal(it["top_idx"][i, :n].cpu().numpy(), order))
        tb = boxes[order]
        want = orc.nms(tb, -np.arange(n, dtype=np.float32), plan.thr)[:plan.post_k]
        c = int(count_h[i])
        ok &= c == len(want) and bool(np.array_equal(it["keep"][i, :c].cpu().numpy(), want))
        ok &= bool(np.array_equal(rois_h[i, :c], tb[want]))
    return bool(ok)


def run_rpn(ctx, args) -> dict:
    torch = ctx.torch
    from faster_rcnn_pytorch_b200 import ops, region, synth
    _lib, lib, dev, world, rank = ctx._lib, ctx.lib, ctx.dev, ctx.world, ctx.rank
    n = synth.num_anchors(HW)
    B = args.batch
    # resident inputs: N_ROTATE different batches, cycled, so each step's 33 MB of inputs is cold in L2
    sets = []
    for r in range(N_ROTATE):
        lg, rg = make_inputs(2000 + 1000 * rank + r, B)
        sets.append((torch.from_numpy(lg).to(dev), torch.from_numpy(rg).to(dev)))
    plan = region.ProposalPlan(B, n, dev, image_hw=HW, mode="train", logits=True, nms_cluster_size=args.nms_cluster)

    def step(i):
        lg, rg = sets[i % N_ROTATE]
        return plan.run(lg, rg)

    for i in range(max(args.warmup, 3)):
        step(i)
    l0 = _lib.launch_count()
    step(0)
    launches_per_step = _lib.launch_count() - l0          # kernels of one frr_rpn_proposals call
    # the step as the library is meant to be driven: the one C-ABI call (it neither allocates nor synchronises) is
    # captured once per resident input set and replayed -- one graph launch per step instead of three kernel launches
    graphs = None
    if not args.eager:
        try:
            graphs = [plan.capture(lg, rg) for lg, rg in sets]
        except RuntimeError:
            graphs = None

    def step_graph(i):
        graphs[i % N_ROTATE].replay()

    run_step = step_graph if graphs else step
    for i in range(max(args.warmup, 3)):
        run_step(i)
    ms_one = ctx.timed(run_step, args.steps)
    ms_eager = ctx.timed(step, args.steps) if graphs else ms_one
    # throughput mode (the headline): several batches in flight on their own streams (region.ProposalPipeline), NMS with
    # one CTA per image (least SM time) -- the top-k and NMS kernels leave 84 of the 148 SMs idle at 64 images, which the
    # neighbouring batches' kernels fill.  Every step is still one complete frr_rpn_proposals call on its batch.
    pipe2 = None
    if graphs and not args.single_stream:
        pipe2 = region.ProposalPipeline(B, n, dev, depth=args.pipe_depth, image_hw=HW, mode="train", logits=True)
        for lg, rg in sets:
            pipe2.capture(lg, rg)

        ticket = [None]

        def step_pipe(i):
            lg, rg = sets[i % N_ROTATE]
            ticket[0] = pipe2.submit(lg, rg)

        for i in range(max(args.warmup, 3)):
            step_pipe(i)
        pipe2.drain()
        ms = ctx.timed(step_pipe, args.steps, tail=pipe2.drain)
        last = pipe2.result(ticket[0])
    else:
        ms = ms_one
        last = (plan.rois, plan.count)
    ctx.keep_outputs("rpn", {"rois": last[0], "count": last[1]})
    launches = launches_per_step * args.steps
    value = world * B * args.steps / (ms * 1e-3)

    # ---- parity of the timed path, outside the timed region: first and last image of one batch vs the oracle
    run_step(0)
    torch.cuda.synchronize()
    verified = verify_proposals(plan, plan.rois, plan.count, (0, B - 1)) if rank == 0 else None
    if pipe2 is not None and rank == 0:   # ... and of both plans of the two-stream pipeline, on two consecutive batches
        for t in range(pipe2.depth):
            pipe2.submit(*sets[(3 + t) % N_ROTATE])
        pipe2.drain()
        torch.cuda.synchronize()
        for pj in pipe2.plans:
            verified = verified and verify_proposals(pj, pj.rois, pj.count, (1, B - 2))
    variant = ops.nms_variant(B, PRE_K, THR, POST_K, cluster_size=1 if pipe2 is not None else args.nms_cluster, unit_boxes=True,
                              device=dev)

    # ---- end to end through the public host-buffer API: pinned host inputs -> H2D -> proposal layer -> D2H of
    #      rois + counts, EVERY step; double buffered (copies of step i+1 overlap the kernels of step i) and,
    #      for comparison, fully serialised (submit, wait, read).
    h_in = [(torch.from_numpy(make_inputs(7000 + 1000 * rank + r, B)[0]).pin_memory(),
             torch.from_numpy(make_inputs(7000 + 1000 * rank + r, B)[1]).pin_memory()) for r in range(2)]
    pipe = region.HostProposalPipeline(plan, depth=2)
    sink = [0]

    def e2e_pipelined(i):
        t = pipe.submit(h_in[i % 2][0], h_in[i % 2][1], stage=False)
        if t >= 1:
            _, cnt = pipe.result(t - 1)
            sink[0] += int(cnt[0])                    # the caller reads the previous step's result

    def e2e_drain():
        _, cnt = pipe.result(pipe._n - 1)
        sink[0] += int(cnt[0])

    def e2e_serial(i):
        t = pipe.submit(h_in[i % 2][0], h_in[i % 2][1], stage=False)
        _, cnt = pipe.result(t)
        sink[0] += int(cnt[0])

    e2e_steps = args.steps
    for i in range(3):
        e2e_serial(i)
    ms_e2e_serial = ctx.median_ms(e2e_serial, e2e_steps, runs=3)
    for i in range(3):
        e2e_pipelined(i)
    e2e_drain()
    ms_e2e = ctx.median_ms(e2e_pipelined, e2e_steps, runs=5, tail=e2e_drain)
    e2e_value = world * B * e2e_steps / (ms_e2e * 1e-3)

    # the host-side ceiling of that pipeline: the same pinned H2D / D2H traffic on the same streams with no kernel between
    d_l = torch.empty_like(sets[0][0]); d_r = torch.empty_like(sets[0][1])
    h_out = torch.empty((B, POST_K, 4), dtype=torch.float32).pin_memory()
    cstream = torch.cuda.Stream(device=dev)

    def copy_only(i):
        with torch.cuda.stream(cstream):
            d_l.copy_(h_in[i % 2][0], non_blocking=True)
            d_r.copy_(h_in[i % 2][1], non_blocking=True)
            h_out.copy_(plan.rois, non_blocking=True)

    def copy_tail():
        cstream.synchronize()

    ms_copy = ctx.median_ms(copy_only, e2e_steps, runs=3, tail=copy_tail)
    copy_value = world * B * e2e_steps / (ms_copy * 1e-3)

    # ---- per-kernel timing on the launching stream (live, CUDA events): raw C-ABI launches into preallocated
    #      buffers (no allocator in the timed loop), inputs rotated as above
    d_boxes = [torch.empty((B, n, 4), dtype=torch.float32, device=dev) for _ in range(N_ROTATE)]
    d_scores = [torch.empty((B, n), dtype=torch.float32, device=dev) for _ in range(N_ROTATE)]
    d_valid = [torch.empty((B, n), dtype=torch.uint8, device=dev) for _ in range(N_ROTATE)]
    t_idx = [torch.empty((B, PRE_K), dtype=torch.int32, device=dev) for _ in range(N_ROTATE)]
    t_cnt = [torch.empty((B,), dtype=torch.int32, device=dev) for _ in range(N_ROTATE)]
    keep = torch.empty((B, POST_K), dtype=torch.int32, device=dev)
    kcnt = torch.empty((B,), dtype=torch.int32, device=dev)
    rois = torch.empty((B, POST_K, 4), dtype=torch.float32, device=dev)
    minsz = float(np.float32(1.0 / 1000.0))

    def k_decode(i, st):
        r = i % N_ROTATE
        _lib.check(lib.frr_rpn_decode(sets[r][1].data_ptr(), sets[r][0].data_ptr(), 1, None, None, 9, HW[0], HW[1], 16,
                                      minsz, d_boxes[r].data_ptr(), d_scores[r].data_ptr(), d_valid[r].data_ptr(), B, n,
                                      st), "frr_rpn_decode")

    def k_topk(i, st):
        r = i % N_ROTATE
        _lib.check(lib.frr_topk_desc_opt(d_scores[r].data_ptr(), d_valid[r].data_ptr(), None, B, n, PRE_K,
                                         None, t_idx[r].data_ptr(), None, None, t_cnt[r].data_ptr(),
                                         1 if nms_cs == 1 else 0, st),     # (the geometry of the timed path)
                   "frr_topk_desc_opt")

    nms_cs = 1 if pipe2 is not None else args.nms_cluster     # the launch geometry of the timed path

    def k_nms(i, st, cs=None):
        r = i % N_ROTATE
        _lib.check(lib.frr_nms_sorted_indirect(d_boxes[r].data_ptr(), n, t_idx[r].data_ptr(), t_cnt[r].data_ptr(), B, PRE_K,
                                               THR, POST_K, keep.data_ptr(), kcnt.data_ptr(), rois.data_ptr(),
                                               nms_cs if cs is None else cs, 1, st),
                   "frr_nms_sorted_indirect")

    reps = max(16, min(args.steps, 64))
    ms_dec = ctx.kernel_ms(k_decode, reps)
    ms_topk = ctx.kernel_ms(k_topk, reps)
    ms_nms = ctx.kernel_ms(k_nms, reps)
    ms_nms_auto = ctx.kernel_ms(lambda i, st: k_nms(i, st, 0), reps)   # automatic geometry: lowest latency of one call
    # single-image NMS latency (whole GPU available to one image: clusters of 8 / 16 CTAs)
    one_src = d_boxes[0][:1].contiguous()
    one_idx = t_idx[0][:1].contiguous()
    one_c = t_cnt[0][:1].contiguous()
    ms_nms1 = {}
    for cs in (8, 16):
        def k_one(i, st, cs=cs):
            _lib.check(lib.frr_nms_sorted_indirect(one_src.data_ptr(), n, one_idx.data_ptr(), one_c.data_ptr(), 1, PRE_K, THR,
                                                   POST_K, keep.data_ptr(), kcnt.data_ptr(), rois.data_ptr(), cs, 1, st),
                       "frr_nms_sorted_indirect")
        ms_nms1[cs] = ctx.kernel_ms(k_one, 50)

    dec_bytes = B * n * 44.0                      # SURVEY §8d: reg 16 + logits 8 + box 16 + score 4 per anchor
    topk_bytes = B * (n * 5.0 + PRE_K * 4.0)      # scores 4 + valid 1 per anchor; sorted index 4 per pick (NMS gathers)
    kern = {"rpn_decode_kernel": ms_dec, "topk_bucket_kernel": ms_topk, "nms_bucket_kernel": ms_nms}
    # SMs a launch occupies (grid / CTAs per SM, capped by the machine): with several batches in flight the step time is
    # the sum of SM time over the kernels / 148, not the sum of the kernel durations
    nsm = ctx.num_sms
    ctas = {"rpn_decode_kernel": nsm, "topk_bucket_kernel": min(B, nsm), "nms_bucket_kernel": min(B * variant["cluster_size"], nsm)}
    sm_ms = {k: kern[k] * ctas[k] for k in kern}
    dominant = max(sm_ms, key=sm_ms.get)
    roof = {
        "rpn_decode_kernel": _hbm_roofline(ctx, "rpn_decode_kernel", dec_bytes, ms_dec,
                                           traffic_note="ncu dram read+write of one launch; below the algorithmic bytes because "
                                                        "the 28 MB of outputs stay in the 126 MB L2 for the top-k / NMS kernels"),
        "topk_bucket_kernel": _hbm_roofline(ctx, "topk_bucket_kernel", topk_bytes, ms_topk),
        "nms_bucket_kernel": _issue_roofline(ctx, "nms_bucket_kernel", ms_nms, sms=ctas["nms_bucket_kernel"]),
    }
    step_ms = ms / args.steps
    line = {
        "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(WORKLOAD, B),
        "config_detail": {"anchors_per_image": n,
                          "l2": f"inputs rotated over {N_ROTATE} resident batches ({N_ROTATE * B * n * 24 / 1e6:.0f} MB > 126 MB L2)"},
        "launch_mode": (f"cuda-graph replay of one frr_rpn_proposals call per step, {args.pipe_depth} steps in flight on "
                        f"{args.pipe_depth} streams, NMS one CTA per image (region.ProposalPipeline)") if pipe2 is not None else
                       ("cuda-graph replay of one frr_rpn_proposals call per step" if graphs else "eager C-ABI call per step"),
        "value_single_stream": world * B * args.steps / (ms_one * 1e-3),
        "value_eager": world * B * args.steps / (ms_eager * 1e-3),
        "verified": verified,
        "verified_how": "images 0 and 63 of a timed batch (single-stream plan) and images 1 and 62 of one batch per plan of "
                        "the multi-stream pipeline: valid mask, top-k order, NMS keep list, count and rois bit-exact "
                        "vs the CPU oracle fed the GPU's decoded boxes (outside the timed region)",
        "nms_variant": variant,
        "nms_us_per_image": 1e3 * ms_nms_auto / B,
        "nms_ms_per_batch_auto_geometry": ms_nms_auto,
        "nms_single_image_latency_us": {f"cluster{cs}": 1e3 * v for cs, v in ms_nms1.items()},
        "kernels_ms_per_batch": kern,
        "kernels_sms_occupied": ctas,
        "kernels_share_of_sm_time": {k: v / sum(sm_ms.values()) for k, v in sm_ms.items()},
        "step_ms_if_sm_time_packed_perfectly": sum(sm_ms.values()) / nsm,
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": pipe.h2d_bytes,
                "d2h_bytes_per_step": pipe.d2h_bytes, "ms_per_step": ms_e2e / e2e_steps,
                "mode": "double-buffered host pipeline (H2D of step i+1 overlaps kernels of step i), median of 5 runs",
                "serialized_value": world * B * e2e_steps / (ms_e2e_serial * 1e-3),
                "host_copy_ceiling": copy_value, "frac_of_host_copy_ceiling": e2e_value / copy_value,
                "host_copy_ceiling_how": "the same pinned H2D (33 MB) + D2H (2 MB) per step on a copy stream, no kernels",
                "host_thread_numa_binding": ctx.numa},
        "gpu_launches": int(launches),
        "roofline": roof[dominant],
        "roofline_other": {k: v for k, v in roof.items() if k != dominant},
        "dominant_kernel": {"kernel": dominant, "share_of_sm_time": sm_ms[dominant] / sum(sm_ms.values())},
    }
    return line


class InFlight:
    """`depth` side streams for throughput timing: step i runs on stream i % depth (steps on one stream stay ordered, steps
    on different streams overlap on the GPU); `begin` orders every side stream after the caller's stream (the timing
    event), `drain` orders the caller's stream after all of them."""

    def __init__(self, torch, dev, depth: int):
        self.torch, self.dev, self.depth = torch, dev, depth
        self.streams = [torch.cuda.Stream(device=dev) for _ in range(depth)]

    def begin(self):
        cur = self.torch.cuda.current_stream(self.dev)
        for st in self.streams:
            st.wait_stream(cur)

    def run(self, i, fn):
        if i == 0:
            self.begin()
        with self.torch.cuda.stream(self.streams[i % self.depth]):
            return fn()

    def drain(self):
        cur = self.torch.cuda.current_stream(self.dev)
        for st in self.streams:
            cur.wait_stream(st)


# ------------------------------------------------------------------------------------------ configs[0] / configs[3]
def _predict_setup(ctx, hw, B, R, NC, seed, n_sets):
    torch = ctx.torch
    from faster_rcnn_pytorch_b200 import region, synth
    dev = ctx.dev
    fh, fw = hw[0] // 16, hw[1] // 16
    n = synth.num_anchors(hw)
    rs = np.random.RandomState(seed + ctx.rank)
    C = 512
    h = dict(
        feats=[rs.standard_normal((B, C, fh, fw)).astype(np.float32) for _ in range(n_sets)],
        lgs=[rs.standard_normal((B, n, 2)).astype(np.float32) for _ in range(n_sets)],
        rgs=[(rs.standard_normal((B, n, 4)) * 0.2).astype(np.float32) for _ in range(n_sets)],
        hcls=rs.standard_normal((B * R, NC)).astype(np.float32),          # head outputs (the FC head is cuBLAS,
        hreg=rs.standard_normal((B * R, 4 * NC)).astype(np.float32))      # not the product)
    d = {k: ([torch.from_numpy(x).to(dev) for x in v] if isinstance(v, list) else torch.from_numpy(v).to(dev))
         for k, v in h.items()}
    plan = region.InferPlan(B, hw, NC, dev)
    return h, d, plan, (fh, fw), n


def _predict_step(ops, fdist, plan, feat, lg, rg, hcls, hreg, fhw, B, R, NC, ids=None, gather=False):
    """FRCNN.predict's region path for a batch (models/model.py:346-402) through region.InferPlan: proposals -> rois5 ->
    RoIPool | per-class decode -> per-class NMS -> packed detections [B,100,6] (+ NCCL all-gather)."""
    pooled, rois, cnt = plan.pool(feat, lg, rg)
    out = plan.detect(hcls, hreg, return_all=True)
    packed, pc = out["packed"], out["count"]
    if gather:
        packed, pc, _ = fdist.gather_detections(packed, pc, ids, equal_batch=True)
    return dict(rois=rois, cnt=cnt, rois5=plan.rois5, pooled=pooled, prob=out["prob"], boxes=out["boxes"], det=out["det"],
                packed=packed, pc=pc)


def verify_predict(out, feat, image: int, R: int, NC: int, fhw) -> bool:
    """One image of the last step against the oracle, stage by stage on the GPU's own inputs: RoIPool max bit-exact on
    the GPU's rois, per-class NMS detections bit-exact on the GPU's probabilities / decoded boxes."""
    from oracle import region_oracle as orc, _cbridge
    _cbridge.load(required=True)
    c = int(out["cnt"][image])
    rois = out["rois"][image, :c].cpu().numpy()
    f = feat[image:image + 1, :32].contiguous().cpu().numpy()                 # 32 of the 512 channels
    want, _ = orc.roi_pool_forward(f, orc.scale_rois(rois, fhw[0], fhw[1]))
    got = out["pooled"][image * R:image * R + c, :32].cpu().numpy()
    ok = bool(np.array_equal(got, want))
    prob = out["prob"].reshape(-1, R, NC)[image, :c].cpu().numpy()
    boxes = out["boxes"].reshape(-1, R, 4 * NC)[image, :c].cpu().numpy()
    wb, wl, ws = orc.suppress(boxes, prob, NC, 0.05)
    db, dl, ds, dc = out["det"]
    k = int(dc[image])
    ok &= k == len(wl) and bool(np.array_equal(db[image, :k].cpu().numpy(), wb)) and \
        bool(np.array_equal(dl[image, :k].cpu().numpy(), wl)) and bool(np.array_equal(ds[image, :k].cpu().numpy(), ws))
    return bool(ok)


def run_predict(ctx, args, which: str) -> dict:
    """configs[0] (`voc1`: 1 image 600x1000, 21 classes, latency) and configs[3] (`infer`: 8 images 800x1333, 81 classes,
    detections all-gathered over NCCL)."""
    torch = ctx.torch
    from faster_rcnn_pytorch_b200 import ops, dist as fdist
    voc = which == "voc1"
    hw, B, R, NC = ((600, 1000), 1, 300, 21) if voc else ((800, 1333), 8, 300, 81)
    NR = 4
    h, d, plan, fhw, n = _predict_setup(ctx, hw, B, R, NC, 9100 if voc else 9000, NR)
    ids = torch.arange(ctx.rank * B, (ctx.rank + 1) * B, dtype=torch.int64, device=ctx.dev)
    keep = {}
    steps = args.steps
    gather = (not voc) and ctx.world > 1

    def step(i, gather=gather):
        r = i % NR
        keep["out"] = _predict_step(ops, fdist, plan, d["feats"][r], d["lgs"][r], d["rgs"][r], d["hcls"], d["hreg"], fhw, B, R, NC,
                                    ids, gather)

    for i in range(max(args.warmup, 3)):
        step(i)
    l0 = ctx._lib.launch_count()
    step(0)
    launches_per_step = ctx._lib.launch_count() - l0
    ms = ctx.timed(step, steps)
    ms_nogather = ctx.timed(lambda i: step(i, False), steps) if gather else ms
    torch.cuda.synchronize()
    verified = verify_predict(keep["out"], d["feats"][(steps - 1) % NR], B - 1, R, NC, fhw) if ctx.rank == 0 else None

    # graph-replayed step (the kernels + torch's allocations are captured once per input set; NCCL stays outside)
    graphs = []
    if not args.eager:
        for r in range(NR):
            g, out = ctx.graph_of(lambda r=r: _predict_step(ops, fdist, plan, d["feats"][r], d["lgs"][r], d["rgs"][r], d["hcls"],
                                                            d["hreg"], fhw, B, R, NC))
            if g is None:
                graphs = []
                break
            graphs.append((g, out))

    def step_graph(i):
        g, out = graphs[i % NR]
        g.replay()
        if gather:
            keep["g"] = fdist.gather_detections(out["packed"], out["pc"], ids, equal_batch=True)

    ms_graph = ctx.timed(step_graph, steps) if graphs else None
    best = min(ms, ms_graph) if ms_graph else ms
    value = ctx.world * B * steps / (best * 1e-3)

    # throughput form (configs[3] only; configs[0] is a latency number): `depth` batches in flight, each on its own stream
    # with its own plan and graphs -- 8 images leave most of the 148 SMs idle in every kernel but RoIPool.  The NCCL gather
    # of a step is issued on the caller's stream once that step's graph has finished (no host synchronisation).
    ms_multi, depth = None, args.pipe_depth
    if graphs and not voc and not args.single_stream:
        from faster_rcnn_pytorch_b200 import region
        fl = InFlight(torch, ctx.dev, depth)
        mg, ok = [], True
        # (kept alive: the graphs hold their buffers; one NMS / top-k CTA per image = the least SM time, as in ProposalPipeline)
        plans = [region.InferPlan(B, hw, NC, ctx.dev, nms_cluster_size=1) for _ in range(depth)]
        keep["plans"] = plans
        for j in range(depth):
            pj = plans[j]
            row = []
            with torch.cuda.stream(fl.streams[j]):
                for r in range(NR):
                    g, out = ctx.graph_of(lambda r=r, pj=pj: _predict_step(ops, fdist, pj, d["feats"][r], d["lgs"][r], d["rgs"][r],
                                                                           d["hcls"], d["hreg"], fhw, B, R, NC))
                    ok &= g is not None
                    row.append((g, out))
            mg.append(row)
        torch.cuda.synchronize()
        if ok:
            done = [torch.cuda.Event() for _ in range(depth)]

            def step_multi(i):
                j = i % depth
                g, out = mg[j][i % NR]

                def go():
                    g.replay()
                    done[j].record()
                fl.run(i, go)
                if gather:
                    torch.cuda.current_stream().wait_event(done[j])
                    keep["g"] = fdist.gather_detections(out["packed"], out["pc"], ids, equal_batch=True)

            for i in range(max(args.warmup, 3)):
                step_multi(i)
            fl.drain()
            ms_multi = ctx.timed(step_multi, steps, tail=fl.drain)
            torch.cuda.synchronize()
            if ctx.rank == 0:   # the last batch every plan produced, against the oracle
                for j in range(min(depth, steps)):
                    i_last = ((steps - 1 - j) // depth) * depth + j
                    verified = bool(verified) and verify_predict(mg[j][i_last % NR][1], d["feats"][i_last % NR], B - 1, R, NC, fhw)
            value = ctx.world * B * steps / (ms_multi * 1e-3)
    # the outputs of the last timed step: in flight, else graph replay, else eager (the same input set in each form)
    last = (mg[(steps - 1) % depth][(steps - 1) % NR][1] if ms_multi else
            graphs[(steps - 1) % NR][1] if graphs else keep["out"])
    arrays = {k: last[k] for k in ("rois", "cnt", "pooled", "prob", "boxes", "packed", "pc")}
    if gather and last is not keep["out"]:   # the graphs hold this rank's detections; the caller receives the gathered ones
        arrays["packed"], arrays["pc"] = keep["g"][0], keep["g"][1]
    ctx.keep_outputs(which, arrays)

    # ---- end to end, strict form: EVERY input of the step from pinned host memory (head outputs, feature map, FC head
    #      outputs), the packed detections read back on the host, every step, serialised (latency form)
    pin = {k: ([torch.from_numpy(x).pin_memory() for x in v] if isinstance(v, list) else torch.from_numpy(v).pin_memory())
           for k, v in h.items()}
    dd = dict(feat=torch.empty_like(d["feats"][0]), lg=torch.empty_like(d["lgs"][0]), rg=torch.empty_like(d["rgs"][0]),
              hcls=torch.empty_like(d["hcls"]), hreg=torch.empty_like(d["hreg"]))
    nrows = B * (ctx.world if gather else 1)
    h_det = torch.empty((nrows, 100, 6), dtype=torch.float32).pin_memory()
    h_cnt = torch.empty((nrows,), dtype=torch.int32).pin_memory()
    sink = [0]

    def e2e_host(i):
        r = i % NR
        dd["feat"].copy_(pin["feats"][r], non_blocking=True)
        dd["lg"].copy_(pin["lgs"][r], non_blocking=True)
        dd["rg"].copy_(pin["rgs"][r], non_blocking=True)
        dd["hcls"].copy_(pin["hcls"], non_blocking=True)
        dd["hreg"].copy_(pin["hreg"], non_blocking=True)
        out = _predict_step(ops, fdist, plan, dd["feat"], dd["lg"], dd["rg"], dd["hcls"], dd["hreg"], fhw, B, R, NC, ids, gather)
        h_det.copy_(out["packed"], non_blocking=True)
        h_cnt.copy_(out["pc"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        sink[0] += int(h_cnt[0])

    def e2e_resident(i):
        # the reference keeps backbone + heads on the device (models/model.py:315,352): only the detections cross PCIe
        if graphs:
            g, out = graphs[i % NR]
            g.replay()
            if gather:
                p, c, _ = fdist.gather_detections(out["packed"], out["pc"], ids, equal_batch=True)
            else:
                p, c = out["packed"], out["pc"]
        else:
            step(i)
            p, c = keep["out"]["packed"], keep["out"]["pc"]
        h_det.copy_(p, non_blocking=True)
        h_cnt.copy_(c, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        sink[0] += int(h_cnt[0])

    for i in range(3):
        e2e_host(i); e2e_resident(i)
    e_steps = steps
    ms_e2e = ctx.median_ms(e2e_host, e_steps, runs=3)
    ms_e2r = ctx.median_ms(e2e_resident, e_steps, runs=3)
    # the same with `depth` batches in flight: the detections of step i - depth are consumed on the host while steps
    # i - depth + 1 .. i run; every step still copies its packed detections + counts into pinned memory
    ms_e2f = None
    if ms_multi:
        hd_ = [torch.empty((nrows, 100, 6), dtype=torch.float32).pin_memory() for _ in range(depth)]
        hc_ = [torch.empty((nrows,), dtype=torch.int32).pin_memory() for _ in range(depth)]
        evs = [torch.cuda.Event() for _ in range(depth)]
        live = [False] * depth

        def consume(j):
            if live[j]:
                evs[j].synchronize()
                sink[0] += int(hc_[j][0])
                live[j] = False

        def e2e_flight(i):
            j = i % depth
            consume(j)                                   # the host reads the result of the step that used this slot
            g, out = mg[j][i % NR]

            def go():
                g.replay()
                done[j].record()
            fl.run(i, go)
            cur = torch.cuda.current_stream()
            cur.wait_event(done[j])
            if gather:
                p, c, _ = fdist.gather_detections(out["packed"], out["pc"], ids, equal_batch=True)
            else:
                p, c = out["packed"], out["pc"]
            hd_[j].copy_(p, non_blocking=True)
            hc_[j].copy_(c, non_blocking=True)
            evs[j].record(cur)
            live[j] = True

        def e2e_flight_tail():
            for j in range(depth):
                consume(j)

        for i in range(2 * depth):
            e2e_flight(i)
        e2e_flight_tail()
        ms_e2f = ctx.median_ms(e2e_flight, e_steps, runs=3, tail=e2e_flight_tail)
    h2d = sum(int(np.prod(x.shape)) * 4 for x in (h["feats"][0], h["lgs"][0], h["rgs"][0], h["hcls"], h["hreg"]))
    d2h = nrows * 100 * 6 * 4 + nrows * 4
    pooled_bytes = B * 512 * fhw[0] * fhw[1] * 4 + B * R * 512 * 49 * 4
    ms_pool = ctx.kernel_ms(lambda i, st: ops.roi_pool_forward(d["feats"][i % NR], keep["out"]["rois5"], want_argmax=False), 8)
    res = {
        "value": value, "unit": "images/s", "ms_per_step": (ms_multi or best) / steps, "steps": steps,
        "latency_us_per_step": 1e3 * best / steps,
        "config": config_of(W_VOC1 if voc else W_INFER, B),
        "config_detail": {"l2": f"inputs rotated over {NR} resident sets"},
        "launch_mode": (f"cuda-graph replay of the region path, {depth} batches in flight on {depth} streams" if ms_multi else
                        "cuda-graph replay of the region path" if (ms_graph and ms_graph <= ms) else "eager ops calls"),
        "ms_per_step_eager": ms / steps, "ms_per_step_graph": (ms_graph / steps) if ms_graph else None,
        "ms_per_step_in_flight": (ms_multi / steps) if ms_multi else None,
        "value_single_stream": ctx.world * B * steps / (best * 1e-3),
        "gpu_launches_per_step": int(launches_per_step), "verified": verified,
        "verified_how": "last image of the last step: RoIPool max (32 channels) and the per-class NMS detections bit-exact vs the "
                        "CPU oracle on the GPU's own rois / probabilities / decoded boxes",
        "e2e": {"value": ctx.world * B * e_steps / (ms_e2e * 1e-3), "unit": "images/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / e_steps,
                "mode": "every input of the step (RPN head outputs, 512-ch feature map, FC head outputs) from pinned host memory, "
                        "packed detections read back, serialised, median of 3 runs"},
        "e2e_resident": {"value": ctx.world * B * e_steps / (ms_e2r * 1e-3), "unit": "images/s", "h2d_bytes_per_step": 0,
                         "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2r / e_steps,
                         "mode": "backbone / head outputs resident on the device as in the reference (models/model.py:315,352), "
                                 "packed detections [B,100,6] + counts read back on the host every step"},
        "e2e_resident_in_flight": ({"value": ctx.world * B * e_steps / (ms_e2f * 1e-3), "unit": "images/s", "h2d_bytes_per_step": 0,
                                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2f / e_steps,
                                    "mode": f"the same, {depth} batches in flight: the host consumes the detections of step i - {depth} "
                                            "while the next steps run"} if ms_e2f else None),
        "roofline": _hbm_roofline(ctx, "roi_pool_fwd_flat_kernel", pooled_bytes, ms_pool,
                                  note="RoIPool forward without argmax: features once + pooled output once"),
        "detections_last_step": int(keep["out"]["pc"].sum()),
    }
    if gather:
        res["collective"] = {"what": "NCCL all_gather_into_tensor of [B,100,6] fp32 + int32 counts + int64 ids (replaces the "
                                     "pickled all_gather of util/misc.py:89-129)",
                             "bytes_per_rank": B * 100 * 6 * 4 + B * 4 + B * 8,
                             "ms_per_step_with": ms / steps, "ms_per_step_without": ms_nogather / steps,
                             "exposed_ms_per_step": max(0.0, (ms - ms_nogather) / steps)}
    return res


# ------------------------------------------------------------------------------------------ configs[2]
def run_train(ctx, args) -> dict:
    torch = ctx.torch
    from faster_rcnn_pytorch_b200 import ops, region, synth, targets
    dev, rank, world = ctx.dev, ctx.rank, ctx.world
    hw, B, G, per, C = (600, 1000), 16, 8, 128, 512
    fh, fw = hw[0] // 16, hw[1] // 16
    n = synth.num_anchors(hw)
    rs = np.random.RandomState(9000 + rank)
    NR = 3   # rotated input sets: 3 x (75 MB features + 206 MB grad_out) > L2
    feats = [torch.from_numpy(rs.standard_normal((B, C, fh, fw)).astype(np.float32)).to(dev) for _ in range(NR)]
    gouts = [torch.from_numpy(rs.standard_normal((B * per, C, 7, 7)).astype(np.float32)).to(dev) for _ in range(NR)]
    lg = torch.from_numpy(rs.standard_normal((B, n, 2)).astype(np.float32)).to(dev)
    rg = torch.from_numpy((rs.standard_normal((B, n, 4)) * 0.2).astype(np.float32)).to(dev)
    gt_h = np.stack([synth.gt_boxes(3000 + 100 * rank + i, G)[0] for i in range(B)])
    lab_h = np.stack([synth.gt_boxes(3000 + 100 * rank + i, G)[1] for i in range(B)])
    gt, lab = torch.from_numpy(gt_h).to(dev), torch.from_numpy(lab_h).to(dev)
    props, pcnt = region.rpn_proposals(lg, rg, image_hw=hw, mode="train")     # config-2 pipeline proposals
    torch.manual_seed(3000 + rank)
    gen = targets.DeviceGenerator(dev) if args.sampling == "device" else None    # torch's mt19937 stream on the device
    stats = {}
    steps = args.steps

    def step(i, gt=gt, lab=lab):
        # device sampling: 6 kernels, no host synchronisation; host sampling: 4 kernels + ONE D2H of counts
        t = targets.make_targets(gt, None, lab, props, pcnt, image_hw=hw, generator=gen)
        ns = t["n_samples"] if isinstance(t["n_samples"], torch.Tensor) else None
        rois5 = ops.rois5(t["sample_rois"], ns, (fh, fw))
        out, arg = ops.roi_pool_forward(feats[i % NR], rois5)
        gin = ops.roi_pool_backward(gouts[i % NR], arg, rois5, feats[0].shape)
        stats["last"] = (out, gin, rois5, arg, t, i % NR)
        return gin

    for i in range(max(args.warmup, 3)):
        step(i)
    l0 = ctx._lib.launch_count()
    step(0)
    launches_per_step = ctx._lib.launch_count() - l0
    ms_one = ctx.timed(step, steps)
    torch.cuda.synchronize()
    gen2 = targets.DeviceGenerator(dev)
    ms_td = ctx.timed(lambda i: targets.make_targets(gt, None, lab, props, pcnt, image_hw=hw, generator=gen2), 12) / 12
    ms_th = ctx.timed(lambda i: targets.make_targets(gt, None, lab, props, pcnt, image_hw=hw), 12) / 12

    # throughput form: `depth` batches in flight on their own streams (each with its own device generator: the sampling
    # stream of a batch is serial, 75 us on one CTA, and the target makers run small grids -- the RoIPool kernels of the
    # neighbouring batch fill the machine meanwhile)
    ms, depth = ms_one, args.pipe_depth
    if not args.single_stream and args.sampling == "device":
        fl = InFlight(torch, dev, depth)
        tplans, tg = [], []
        gt_j = [gt.clone() for _ in range(depth)]      # per-slot ground truth (the end-to-end form refills it every step)
        lab_j = [lab.clone() for _ in range(depth)]
        for j in range(depth):
            with torch.cuda.stream(fl.streams[j]):
                pj = region.TrainPlan(B, hw, dev, generator=targets.DeviceGenerator(dev))
                row = []
                for r in range(NR):
                    # the two halves of the step as CUDA graphs (the head's forward / backward sits between them in a real
                    # step): targets + rois5 + RoIPool forward, then RoIPool backward on that forward's argmax
                    g1, o1 = pj.capture_targets_and_pool(feats[r], gt_j[j], lab_j[j], props, pcnt)
                    last = dict(pj.last)
                    g2, o2 = pj.capture_pool_backward(gouts[r])
                    row.append((g1, g2, o1, o2, last))
            tplans.append(pj)
            tg.append(row)
        torch.cuda.synchronize()

        def step_multi(i):
            j, r = i % depth, i % NR

            def go():
                g1, g2, o1, o2, last = tg[j][r]
                g1.replay()
                g2.replay()
                stats["last"] = (o1[1], o2, tplans[j].rois5, last["argmax"], o1[0], r)
            fl.run(i, go)

        for i in range(max(args.warmup, 3)):
            step_multi(i)
        fl.drain()
        ms = ctx.timed(step_multi, steps, tail=fl.drain)
        torch.cuda.synchronize()
    out, gin, rois5, arg, t, r_last = stats["last"]
    ctx.keep_outputs("train", dict(t, rois5=rois5, pooled=out, argmax=arg, grad_features=gin))

    verified = None
    if rank == 0:   # image 0 of the last step: RoIPool forward (max + argmax) bit-exact, backward within 1e-5 of max|grad|
        from oracle import region_oracle as orc, _cbridge
        _cbridge.load(required=True)
        r5 = rois5[:per].cpu().numpy()
        live = r5[:, 0] >= 0
        f = feats[r_last][:1, :16].contiguous().cpu().numpy()
        wo, wa = orc.roi_pool_forward(f, r5[live])
        verified = bool(np.array_equal(out[:per][torch.from_numpy(live).to(dev)][:, :16].cpu().numpy(), wo)) and \
            bool(np.array_equal(arg[:per][torch.from_numpy(live).to(dev)][:, :16].cpu().numpy(), wa))
        # labels: the reference's invariants (<= 128 positives, 256 sampled in total when enough candidates)
        lbl = t["rpn_cls"][0].cpu().numpy()
        verified &= int((lbl == 1).sum()) <= 128 and int((lbl >= 0).sum()) == 256

    obytes = B * per * C * 49 * 4
    fbytes = B * C * fh * fw * 4
    ms_f = ctx.kernel_ms(lambda i, st: ops.roi_pool_forward(feats[i % NR], rois5), 12)
    ms_b = ctx.kernel_ms(lambda i, st: ops.roi_pool_backward(gouts[i % NR], arg, rois5, feats[0].shape), 12)
    # ---- end to end: what crosses PCIe in the reference's training step for this stage is the ground truth (boxes +
    #      labels, from the data loader, main.py:66-75) going in and nothing coming out (targets feed the loss on the
    #      device); here the sampled class targets + sample counts are read back every step as the step's result
    h_gt = torch.from_numpy(gt_h).pin_memory()
    h_lab = torch.from_numpy(lab_h).pin_memory()
    d_gt, d_lab = torch.empty_like(gt), torch.empty_like(lab)
    h_cls = torch.empty((B, per), dtype=torch.int64).pin_memory()
    sink = [0]

    def e2e(i):
        d_gt.copy_(h_gt, non_blocking=True)
        d_lab.copy_(h_lab, non_blocking=True)
        step(i, d_gt, d_lab)
        h_cls.copy_(stats["last"][4]["frcnn_cls"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        sink[0] += int(h_cls[0, 0])

    for i in range(3):
        e2e(i)
    e_steps = steps
    ms_e2e = ctx.median_ms(e2e, e_steps, runs=3)
    # the same with `depth` batches in flight (graph replays): H2D of the ground truth into the slot's tensors, both graphs,
    # D2H of the sampled class targets, the host consuming the result of step i - depth
    ms_e2f = None
    if ms is not ms_one:
        h_cls_j = [torch.empty((B, per), dtype=torch.int64).pin_memory() for _ in range(depth)]
        evs = [torch.cuda.Event() for _ in range(depth)]
        live_j = [False] * depth

        def consume(j):
            if live_j[j]:
                evs[j].synchronize()
                sink[0] += int(h_cls_j[j][0, 0])
                live_j[j] = False

        def e2e_flight(i):
            j, r = i % depth, i % NR
            consume(j)

            def go():
                g1, g2, o1, o2, last = tg[j][r]
                gt_j[j].copy_(h_gt, non_blocking=True)
                lab_j[j].copy_(h_lab, non_blocking=True)
                g1.replay()
                g2.replay()
                h_cls_j[j].copy_(o1[0]["frcnn_cls"], non_blocking=True)
                evs[j].record()
            fl.run(i, go)
            live_j[j] = True

        def e2e_flight_tail():
            for j in range(depth):
                consume(j)

        for i in range(2 * depth):
            e2e_flight(i)
        e2e_flight_tail()
        ms_e2f = ctx.median_ms(e2e_flight, e_steps, runs=3, tail=e2e_flight_tail)
    fb = fbytes + 2 * obytes
    return {
        "value": world * B * steps / (ms * 1e-3), "unit": "images/s", "ms_per_step": ms / steps, "steps": steps,
        "value_single_stream": world * B * steps / (ms_one * 1e-3), "ms_per_step_single_stream": ms_one / steps,
        "launch_mode": (f"cuda-graph replays (targets + RoIPool forward | RoIPool backward), {depth} batches in flight on "
                        f"{depth} streams" if ms is not ms_one else "eager ops calls, one batch at a time"),
        "config": config_of(W_TRAIN, B),
        "config_detail": {"l2": f"features / grad_out rotated over {NR} resident sets (> 126 MB L2)"},
        "kernels_ms_per_batch": {"roi_pool_fwd": ms_f, "roi_pool_bwd": ms_b,
                                 "make_targets(device sampling: 6 kernels, no sync)": ms_td,
                                 "make_targets(host sampling: 4 kernels + D2H + randperm + H2D)": ms_th},
        "sampling": args.sampling, "gpu_launches_per_step": int(launches_per_step), "verified": verified,
        "verified_how": "image 0 of the last step: RoIPool max + argmax (16 channels) bit-exact vs the CPU oracle on the GPU's "
                        "sampled rois; sampling invariants of the RPN labels",
        "e2e": {"value": world * B * e_steps / (ms_e2e * 1e-3), "unit": "images/s",
                "h2d_bytes_per_step": int(gt_h.nbytes + lab_h.nbytes), "d2h_bytes_per_step": B * per * 8,
                "ms_per_step": ms_e2e / e_steps,
                "mode": "ground-truth boxes + labels from pinned host memory, sampled class targets read back, every step, "
                        "serialised; features / grad_out resident (backbone and head backward run on the device, "
                        "models/model.py:315)"},
        "e2e_in_flight": ({"value": world * B * e_steps / (ms_e2f * 1e-3), "unit": "images/s",
                           "h2d_bytes_per_step": int(gt_h.nbytes + lab_h.nbytes), "d2h_bytes_per_step": B * per * 8,
                           "ms_per_step": ms_e2f / e_steps,
                           "mode": f"the same copies every step, {depth} batches in flight (graph replays), the host consumes the "
                                   f"result of step i - {depth}"} if ms_e2f else None),
        "roofline": _hbm_roofline(ctx, "roi_pool_fwd_flat_kernel", fb, ms_f),
        "roofline_bwd": _hbm_roofline(ctx, "roi_pool_bwd_color_kernel", fb, ms_b),
    }


# ------------------------------------------------------------------------------------------ configs[4]
def run_joint(ctx, args) -> dict:
    """Approximate joint training step, 4 images/GPU at 600x1000: VGG16 backbone + FC head on torch / cuDNN / cuBLAS under DDP
    (NCCL all-reduce of the 548 MB of fp32 gradients), region stage = libfrr."""
    torch = ctx.torch
    from faster_rcnn_pytorch_b200 import targets
    sys.path.insert(0, os.path.join(REPO, "tools"))
    import frcnn_harness as fh_
    dev, rank, world, local = ctx.dev, ctx.rank, ctx.world, ctx.local
    hw, B, G = (600, 1000), 4, 8
    torch.manual_seed(1234)
    model = fh_.FRCNNTrain(21).to(dev).to(memory_format=torch.channels_last)
    net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local]) if world > 1 else model
    opt = torch.optim.SGD(net.parameters(), lr=1e-3, momentum=0.9)
    torch.manual_seed(4000 + rank)
    gen = targets.DeviceGenerator(dev)
    batches = [fh_.make_batch(B, hw, G, dev, seed=10 * rank + i) for i in range(3)]
    kept = {}

    def step(i):
        x, gt, lab = batches[i % 3]
        opt.zero_grad(set_to_none=True)
        loss = net(x, gt, lab, gen)
        loss[:, 0].mean().backward()
        opt.step()
        kept["loss"] = loss
        return loss

    for i in range(max(args.warmup, 3)):
        step(i)
    l0 = ctx._lib.launch_count()
    ms = ctx.timed(step, args.steps)
    launches = ctx._lib.launch_count() - l0
    ctx.keep_outputs("joint", {"loss": kept["loss"]})
    model.timer.enabled = True
    for i in range(4):
        step(i)
    region_ms = model.timer.total_ms() / 4          # forward-side region calls (their backward runs inside autograd)
    model.timer.enabled = False
    last = step(0).detach().cpu().numpy()
    return {
        "metric": METRIC, "value": world * B * args.steps / (ms * 1e-3), "unit": "images/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[4]: approximate joint training step (fwd + bwd + SGD), VGG16 Faster R-CNN, 4 images/GPU "
                               "at 600x1000, G=8; backbone/heads torch+cuDNN under DDP (NCCL), region stage libfrr",
                   "images_per_gpu_per_step": B, "parallelism": f"dp{world}"},
        "region_stage_forward_ms_per_step": region_ms, "region_stage_share": region_ms / (ms / args.steps),
        "loss_last_step": [float(v) for v in last.mean(axis=0)], "gpu_launches": int(launches)}


def _as_line(ctx, args, res: dict) -> dict:
    """A sub-result printed on its own (`--workload voc1|train|infer`) in the line format of the contract."""
    line = {"metric": METRIC, "n_gpus": ctx.world, "warmup": max(args.warmup, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
    line.update(res)
    line["gpu_launches"] = int(res.get("gpu_launches_per_step", 0)) * int(res.get("steps", 0))
    return line


def run_ours(args):
    ctx = Ctx(dump=args.dump_outputs is not None)
    sampler = ClockSampler(ctx.local) if ctx.rank == 0 else None
    threads = os.cpu_count() or 1
    want_cpu = ctx.rank == 0 and ctx.world == 1 and not args.no_cpu
    if args.workload == "joint":
        line = run_joint(ctx, args)
    elif args.workload in ("voc1", "infer", "train"):
        res = run_train(ctx, args) if args.workload == "train" else run_predict(ctx, args, args.workload)
        line = _as_line(ctx, args, res)
        if want_cpu:
            line["cpu_baseline"] = cpu_baseline(args.workload, threads)
    else:
        line = run_rpn(ctx, args)
        if args.workload == "all":
            sub = {}
            for name in ("voc1", "train", "infer"):
                sub[name] = run_train(ctx, args) if name == "train" else run_predict(ctx, args, name)
            line["sub_results"] = sub
        clocks = sampler.stop() if sampler else None
        sampler = None
        line["clocks"] = clocks
        if want_cpu:   # bounded samples of the same workloads on the host cores (rank 0, N = 1 only)
            line["cpu_baseline"] = cpu_baseline("rpn", threads, per_thread=4)
            for name in line.get("sub_results", {}):
                line["sub_results"][name]["cpu_baseline"] = cpu_baseline(name, threads)
        else:
            line["cpu_baseline"] = None
    if sampler is not None:
        line["clocks"] = sampler.stop()
    if ctx.rank == 0:
        print(json.dumps(line), flush=True)
    ctx.close()
    if ctx.dump:   # after the result line: an oversized dump must not cost the measurement
        write_outputs(ctx.dumps, args.dump_outputs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--eager", action="store_true", help="time eager C-ABI calls instead of CUDA-graph replays")
    ap.add_argument("--single-stream", action="store_true", help="rpn workload: one step at a time on one stream")
    ap.add_argument("--nms-cluster", type=int, default=0, help="rpn workload, single-stream plan: NMS CTAs per image (0 = auto)")
    ap.add_argument("--pipe-depth", type=int, default=4, help="rpn workload: batches in flight (region.ProposalPipeline)")
    ap.add_argument("--sampling", default="device", choices=["device", "host"],
                    help="train workload: where the reference's torch.randperm draws are replayed")
    ap.add_argument("--workload", default="all", choices=["all", "rpn", "voc1", "train", "infer", "joint"],
                    help="all = configs[1] headline + sub_results for configs[0], [2], [3] (the driver's line); rpn = configs[1] "
                         "only; voc1 = configs[0]; train = configs[2]; infer = configs[3]; joint = configs[4]")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs of every workload run to DIR/<workload>_<output>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
