"""Developer tool: the bucketed NMS with one CTA per image at two CTAs per SM, against a parent build (GPU box).

    python tools/nms_two_per_sm.py kernel
        per-launch time of the automatic one-CTA-per-image NMS (12 000 -> 2 000 @ 0.7) over B = 64, 128, 148 and 296
        images, from CUDA-graph replays over 8 rotated input sets (as bench.py times it), for the tree this file is in.
    python tools/nms_two_per_sm.py compare --parent DIR --out DIR [--runs 3] [--kernel-rounds 2]
        the same kernel timings and `bench.py --gpus 1` alternately in this tree and in the built tree DIR (the parent
        commit), the occupancy of every bucketed NMS kernel, and a byte comparison of both trees' --dump-outputs.
Every result is one JSON line, printed and appended to OUT/nms_two_per_sm.jsonl, with the card, power limit and clocks.
"""
import argparse
import glob
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THR, PRE_K, POST_K = 0.7, 12000, 2000
N_ROTATE = 8


def kernel_times():
    sys.path.insert(0, ROOT)
    import torch
    from faster_rcnn_pytorch_b200 import _lib, ops, synth
    lib = _lib.load()
    dev = torch.device("cuda:0")
    hw = (608, 1008)
    n = synth.num_anchors(hw)
    bmax = 296
    g = torch.Generator(device=dev)
    sets = []
    for r in range(N_ROTATE):  # bench.py's input statistics, drawn on the device
        g.manual_seed(100 + r)
        logits = torch.randn((bmax, n, 2), generator=g, device=dev)
        reg = torch.randn((bmax, n, 4), generator=g, device=dev) * 0.2
        boxes, scores, valid = ops.rpn_decode(reg, logits, image_hw=hw)
        top = ops.topk_desc(scores, PRE_K, valid=valid)
        sets.append((boxes, top["idx"].contiguous(), top["count"].contiguous()))
        del logits, reg, scores, valid
    keep = torch.empty((bmax, POST_K), dtype=torch.int32, device=dev)
    kcnt = torch.empty((bmax,), dtype=torch.int32, device=dev)
    rois = torch.empty((bmax, POST_K, 4), dtype=torch.float32, device=dev)
    out = []
    for B in (64, 128, 148, 296):
        v = ops.nms_variant(B, PRE_K, THR, POST_K, cluster_size=1, unit_boxes=True)
        views = [(b[:B], i[:B].contiguous(), c[:B].contiguous()) for b, i, c in sets]

        def launch(k, st):
            b, i, c = views[k % N_ROTATE]
            _lib.check(lib.frr_nms_sorted_indirect(b.data_ptr(), n, i.data_ptr(), c.data_ptr(), B, PRE_K, THR, POST_K,
                                                   keep.data_ptr(), kcnt.data_ptr(), rois.data_ptr(), 1, 1, st),
                       "frr_nms_sorted_indirect")

        st = torch.cuda.current_stream().cuda_stream
        for k in range(N_ROTATE):
            launch(k, st)
        torch.cuda.synchronize()
        reps = 32
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, capture_error_mode="thread_local"):
            cs = torch.cuda.current_stream().cuda_stream
            for k in range(reps):
                launch(k, cs)
        graph.replay()
        torch.cuda.synchronize()
        us = []
        for _ in range(7):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graph.replay()
            e1.record()
            torch.cuda.synchronize()
            us.append(1e3 * e0.elapsed_time(e1) / reps)
        us.sort()
        out.append({"what": "nms_kernel", "tree": ROOT, "B": B, "variant": v, "us_per_launch_median": us[len(us) // 2],
                    "us_per_launch_min": us[0], "us_per_launch_max": us[-1], "us_per_image": us[len(us) // 2] / B})
        del graph
    return out


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else r.stderr.strip()


def emit(out_dir, rec):
    rec = dict(rec, card=card())
    line = json.dumps(rec)
    print(line, flush=True)
    if out_dir:
        with open(os.path.join(out_dir, "nms_two_per_sm.jsonl"), "a") as f:
            f.write(line + "\n")


def run_json_lines(cmd, cwd):
    r = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"{' '.join(cmd)} in {cwd} failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}")
    return [json.loads(x) for x in r.stdout.splitlines() if x.startswith("{")]


def occupancy(tmp):
    exe = os.path.join(tmp, "nms_occupancy")
    csrc = os.path.join(ROOT, "faster_rcnn_pytorch_b200", "csrc")
    subprocess.run([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), "-gencode", "arch=compute_100a,code=sm_100a",
                    "-O3", "-std=c++17", "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
                    "-I", os.path.join(ROOT, "include"), "-I", csrc, "-o", exe,
                    os.path.join(ROOT, "tools", "nms_occupancy.cu")], check=True)
    return run_json_lines([exe], ROOT)


def compare(args):
    os.makedirs(args.out, exist_ok=True)
    trees = {"parent": os.path.abspath(args.parent), "change": ROOT}
    # the parent commit has no copy of this tool
    me = os.path.abspath(__file__)
    with tempfile.TemporaryDirectory() as tmp:
        for name, tree in trees.items():
            subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.build()"], cwd=tree, check=True)
        for rec in occupancy(tmp):
            emit(args.out, dict(rec, what="occupancy"))
        for rnd in range(args.kernel_rounds):
            for name, tree in trees.items():
                for rec in run_json_lines([sys.executable, me, "kernel", "--root", tree], tree):
                    emit(args.out, dict(rec, build=name, round=rnd))
        dumps = {}
        for rnd in range(args.runs):
            for name, tree in trees.items():
                cmd = [sys.executable, "bench.py", "--gpus", "1"]
                if rnd == 0:
                    dumps[name] = os.path.join(tmp, "dump_" + name)
                    cmd += ["--dump-outputs", dumps[name]]
                for rec in run_json_lines(cmd, tree):
                    keep = {k: rec.get(k) for k in ("value", "value_single_stream", "nms_ms_per_batch_auto_geometry",
                                                    "nms_single_image_latency_us", "verified", "nms_variant",
                                                    "kernels_ms_per_batch")}
                    keep["sub_results"] = {name: {k: s.get(k) for k in ("value", "unit", "verified")}
                                           for name, s in rec.get("sub_results", {}).items()}
                    emit(args.out, dict(keep, what="bench", build=name, round=rnd))
        a, b = (sorted(os.path.relpath(p, dumps[k]) for p in glob.glob(os.path.join(dumps[k], "*.npy")))
                for k in ("parent", "change"))
        same = {f: open(os.path.join(dumps["parent"], f), "rb").read() == open(os.path.join(dumps["change"], f), "rb").read()
                for f in a if f in b}
        emit(args.out, {"what": "dump_outputs", "files_parent": a, "files_change": b, "identical": same,
                        "all_identical": a == b and all(same.values())})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("mode", choices=["kernel", "compare"])
    ap.add_argument("--root", help="kernel mode: the tree whose build is timed (default: this file's tree)")
    ap.add_argument("--parent")
    ap.add_argument("--out")
    ap.add_argument("--runs", type=int, default=3, help="compare: bench.py runs per build")
    ap.add_argument("--kernel-rounds", type=int, default=2, help="compare: kernel timing rounds per build")
    args = ap.parse_args()
    if args.mode == "kernel":
        global ROOT
        if args.root:
            ROOT = os.path.abspath(args.root)
        for rec in kernel_times():
            print(json.dumps(rec), flush=True)
    else:
        compare(args)


if __name__ == "__main__":
    main()
