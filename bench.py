#!/usr/bin/env python
"""bench.py — headline benchmark of the YOLOv3 hot path on B200 (contract: see task ④).

Workload (BASELINE.json configs[1]): batch=64 416x416 inference, 80 classes, one step =
forward (75 convs) -> decode (+ score = conf*prob) -> per-image gpu_nms(max_boxes=200,
score_thresh=0.3, nms_thresh=0.45) over one batch of synthetic images.  Weights are random
(no checkpoint is shipped): SURVEY.md §8d cfg 2 — Glorot init, detection-head weights x8
and conf bias -2 so that scores straddle the 0.3 threshold.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--size S]
                  [--dump-outputs DIR]

Every timed loop runs exactly K steps.  --dump-outputs writes the detections of the last timed device-resident step
(rank 0) to DIR/<name>.npy; the inputs and weights are seeded, so two builds run with the same arguments can be
compared array for array.

`value`  : images/s with the batch already resident in HBM, CUDA-event timed, max over ranks.
`e2e`    : images/s through the public API from pinned HOST float32 images (H2D inside the
           timed region) to host-side detections (D2H inside the timed region).
`roofline`: the tensor-core conv kernel (74 launches/step): algorithmic conv FLOPs / event-timed
           duration of those launches, against MEASURED_PEAKS.json's sustained bf16 peak.
`cpu_baseline` / `--impl reference`: the CPU oracle port (TensorFlow 1.x cannot be installed in
           this image) timed on the host cores on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

NMS_ARGS = dict(max_boxes=200, score_thresh=0.3, nms_thresh=0.45)   # test_single_image.py:57
CLASS_NUM = 80
FWD_GFLOP_416 = 65.864075264       # SURVEY.md Appendix A (2*MAC, 75 convs, per image @416^2)
STEM_GFLOP_416 = 2 * 416 * 416 * 32 * 27 / 1e9


def make_bench_params(seed=2, specs=None):
    """SURVEY.md §8d cfg 2 parameters (numpy, HWIO): Glorot-uniform, identity BN, head x8, conf bias -2.
    `specs`: (cin, cout, k, stride, has_bn) per conv.  The CPU arm passes nothing and walks the ORACLE's layer list, so it
    never imports the product package; the GPU arm passes the product's own yolov3.conv_table(), so it never imports
    oracle/ (same table, same RNG stream: tests/test_bench_contract.py checks the two agree)."""
    if specs is None:
        from oracle import yolov3_oracle as O
        specs = [(cin, cout, k, s, bn) for _scope, cin, cout, k, s, bn in O.conv_specs(CLASS_NUM)]
    rng = np.random.default_rng(seed)
    ps = []
    for cin, cout, k, s, bn in specs:
        lim = np.sqrt(6.0 / (k * k * (cin + cout)))
        w = rng.uniform(-lim, lim, (k, k, cin, cout)).astype(np.float32)
        if bn:
            ps.append(dict(w=w, gamma=np.ones(cout, np.float32), beta=np.zeros(cout, np.float32),
                           mean=np.zeros(cout, np.float32), var=np.ones(cout, np.float32)))
        else:
            b = np.zeros(cout, np.float32)
            b.reshape(3, -1)[:, 4] = -2.0
            ps.append(dict(w=(w * 8.0).astype(np.float32), b=b))
    return ps


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                f = [v.strip() for v in out.split(",")]
                self.samples.append((float(f[0]), float(f[1])))
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(s[0] for s in self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.samples[0][1], "reasons": sorted(self.reasons),
                "samples": len(sm)}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(tflops=p.get("bf16_tflops_sustained", p.get("bf16_tflops")), hbm=p.get("hbm_gbs"), src="measured (MEASURED_PEAKS.json, sustained bf16)")
    return dict(tflops=1400.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


# --------------------------------------------------------------------------------------
# CPU reference arm (oracle port; TensorFlow is not installable here)
# --------------------------------------------------------------------------------------
def cpu_step(O, x, params, anchors):
    """One reference-path pass on the host: forward -> predict -> score -> per-image gpu_nms."""
    fms = O.forward(x, params)
    boxes, confs, probs = O.predict(fms, anchors, x.shape[1:3], CLASS_NUM)
    scores = confs * probs
    k = 0
    for i in range(x.shape[0]):
        r = O.gpu_nms_c(boxes[i:i + 1], scores[i:i + 1], CLASS_NUM, NMS_ARGS["max_boxes"], NMS_ARGS["score_thresh"],
                        NMS_ARGS["nms_thresh"])     # C restatement of TF's single-threaded CPU kernel
        k += len(r[1])
    return k


CPU_IMAGES_PER_WORKER = int(os.environ.get("YB_CPU_IMAGES", "8"))   # images every worker processes per pass (in batches of CPU_BATCH)
CPU_BATCH = 4
CPU_SKIP_SECONDS = 75.0        # a thread configuration projected to need longer than this is listed, not run


def _cpu_worker(size, passes, warmup, images, threads):
    """One CPU worker process: `warmup` + `passes` passes over `images` images with `threads` torch threads.
    Prints {"pass_seconds": [...]} (timed passes only).  Imports the oracle only — never the product package."""
    import torch
    from oracle import yolov3_oracle as O
    torch.set_num_threads(threads)
    params = make_bench_params()
    x = np.random.default_rng(2).random((images, size, size, 3), dtype=np.float32)
    times = []
    for it in range(warmup + passes):
        t0 = time.perf_counter()
        for lo in range(0, images, CPU_BATCH):
            cpu_step(O, x[lo:lo + CPU_BATCH], params, O.COCO_ANCHORS)
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return times


def _run_candidate(size, workers, threads, passes, warmup, images):
    """`workers` concurrent worker processes x `threads` threads -> (images/s, per-worker pass times)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--cpu-worker", f"{size},{passes},{warmup},{images},{threads}"]
    env = dict(os.environ, OMP_NUM_THREADS=str(threads), MKL_NUM_THREADS=str(threads), CUDA_VISIBLE_DEVICES="")
    procs = [subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, env=env) for _ in range(workers)]
    t_all = []
    try:
        for pr in procs:
            out = pr.communicate(timeout=1200)[0].strip().splitlines()
            t_all.append(json.loads(out[-1])["pass_seconds"])
    except Exception as e:
        for pr in procs:
            if pr.poll() is None:
                pr.kill()
        return None, f"worker failed: {e}"
    # every worker processed images*passes images; the job is done when the slowest worker is
    total = max(sum(t) for t in t_all)
    return workers * images * len(t_all[0]) / total, t_all


def run_cpu(size, passes=3, warmup=1):
    """The reference path's CPU port on the host cores — a MEASUREMENT, not a lottery:
    a fixed sweep of thread configurations (1 x all cores, cores/16 x 16 threads, cores/32 x 32 threads), every one
    run in worker subprocesses with the same code, CPU_IMAGES_PER_WORKER images per worker per pass, `passes` timed
    passes after `warmup` passes; the reported value is the best configuration's, with every candidate listed.  A 2-image
    probe only decides whether a configuration is too slow to be worth its full run (it is then listed as skipped).
    Used verbatim by `--impl reference` and by the `cpu_baseline` leg of the GPU arm."""
    ncpu = os.cpu_count() or 1
    cands = []
    for w, t in ((1, ncpu), (max(1, ncpu // 16), min(16, ncpu)), (max(1, ncpu // 32), min(32, ncpu))):
        if (w, t) not in cands:
            cands.append((w, t))
    forced = os.environ.get("YB_CPU_THREADS")
    if forced:
        t = max(1, min(ncpu, int(forced)))
        cands = [(max(1, ncpu // t), t)]
    listing, best = [], None
    for w, t in cands:
        probe, _ = _run_candidate(size, w, t, 1, 1, 2)
        entry = {"workers": w, "threads": t, "probe_images_per_s": probe}
        if probe is None:
            entry["skipped"] = "probe failed"
        else:
            projected = w * CPU_IMAGES_PER_WORKER * (passes + warmup) / probe
            if projected > CPU_SKIP_SECONDS and len(cands) > 1 and (best is not None or (w, t) != cands[-1]):
                entry["skipped"] = f"projected {projected:.0f} s > {CPU_SKIP_SECONDS:.0f} s"
            else:
                val, t_all = _run_candidate(size, w, t, passes, warmup, CPU_IMAGES_PER_WORKER)
                if val is None:
                    entry["skipped"] = t_all
                else:
                    entry["images_per_s"] = val
                    entry["pass_seconds_slowest_worker"] = [round(v, 3) for v in max(t_all, key=sum)]
                    if best is None or val > best[0]:
                        best = (val, w, t, max(sum(tt) for tt in t_all) / len(t_all[0]))
        listing.append(entry)
    if best is None:      # nothing ran in full: fall back to the best probe, and say so
        ok = [e for e in listing if e.get("probe_images_per_s")]
        e = max(ok, key=lambda q: q["probe_images_per_s"])
        best = (e["probe_images_per_s"], e["workers"], e["threads"], 2 * e["workers"] / e["probe_images_per_s"])
    model = ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    val, w, t, per_pass = best
    return dict(value=val, unit="images/s", cores=w * t, kind="port", cpu_model=model, host_cores=ncpu,
                candidates=listing,
                sample=f"best of {len(listing)} fixed thread configurations: {w} worker process(es) x {t} threads, each "
                       f"{passes} timed passes (+{warmup} warm-up) over {CPU_IMAGES_PER_WORKER} images {size}x{size} in batches of "
                       f"{CPU_BATCH} (forward + decode + per-image NMS, fp32; torch-CPU conv2d restatement of the TF1 graph + C "
                       f"restatement of TF's NMS kernel; TensorFlow is not installable in this image)"), per_pass


def nms_stress(pkg, with_cpu, iters):
    """BASELINE.json configs[4]: 100k pre-NMS boxes x 80 classes, gpu_nms(200, 0.3, 0.45); sparse (s=u1*u2, ~5% pass)
    and dense (s~U[0,1), 70% pass) score variants, `iters` timed calls each.  Unit: (box, class) pairs per second = 8e6 / t."""
    import torch
    from tests.synth import gen_nms_boxes
    from yolov3_tensorflow_b200.utils.nms_utils import batched_nms_raw
    out = {}
    for name, dense in (("sparse", False), ("dense", True)):
        b, sc = gen_nms_boxes(5, 100000, CLASS_NUM, dense=dense)
        bd, sd = torch.from_numpy(b[None]).cuda(), torch.from_numpy(sc[None]).cuda()
        for _ in range(3):
            r = batched_nms_raw(bd, sd, CLASS_NUM, **NMS_ARGS)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            r = batched_nms_raw(bd, sd, CLASS_NUM, **NMS_ARGS)
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) / iters * 1e-3
        rec = {"ms": t * 1e3, "pairs_per_s": 8e6 / t, "kept": int(r[4][0]), "candidates": int((sc >= 0.3).sum()),
               "read_gbs": 33.6e6 / t / 1e9}
        if with_cpu:
            from oracle import yolov3_oracle as O
            t0 = time.perf_counter()
            ob = O.gpu_nms_c(b[None], sc[None], CLASS_NUM, NMS_ARGS["max_boxes"], NMS_ARGS["score_thresh"], NMS_ARGS["nms_thresh"])
            tc = time.perf_counter() - t0
            rec["cpu_port_ms"] = tc * 1e3
            rec["cpu_port_pairs_per_s"] = 8e6 / tc
            rec["indices_bit_exact_vs_cpu"] = bool(np.array_equal(ob[3], r[3][0, :len(ob[3])].cpu().numpy()) and len(ob[3]) == int(r[4][0]))
        out[name] = rec
    return out


def synth_gt_lists(rng, n, size, class_num=CLASS_NUM, max_boxes=50):
    """SURVEY.md §8d cfg 3/4 ground truth as LISTS (what a data loader hands over): per image U{1..max} boxes
    [x0, y0, x1, y1, mix-up weight 1], w, h ~ logU[8, 400] clipped to the image, uniform centres and classes."""
    bl, ll = [], []
    for _ in range(n):
        v = int(rng.integers(1, max_boxes + 1))
        wh = np.exp(rng.uniform(np.log(8), np.log(400), (v, 2))).clip(max=size)
        c = rng.uniform(0, size, (v, 2)).clip(wh / 2, size - wh / 2 - 1e-3)
        bl.append(np.concatenate([c - wh / 2, c + wh / 2, np.ones((v, 1))], axis=1).astype(np.float32))
        ll.append(rng.integers(0, class_num, v).astype(np.int64))
    return bl, ll


def synth_y_true(rng, n, size, anchors, class_num=CLASS_NUM, max_boxes=50):
    """SURVEY.md §8d cfg 3/4 targets: per image U{1..50} boxes, w,h ~ logU[8,400], best-anchor assignment
    (utils/data_utils.py:51-115 semantics, vectorised on the host) -> three y_true tensors on the GPU."""
    import torch
    ys = [np.zeros((n, size // s, size // s, 3, 6 + class_num), np.float32) for s in (32, 16, 8)]
    for y in ys:
        y[..., -1] = 1.0
    anc = np.asarray(anchors, np.float32)
    for i in range(n):
        v = int(rng.integers(1, max_boxes + 1))
        wh = np.exp(rng.uniform(np.log(8), np.log(400), (v, 2))).clip(max=size)
        c = rng.uniform(0, size, (v, 2)).clip(wh / 2, size - wh / 2)
        inter = np.minimum(wh[:, None, :], anc[None]).prod(-1)
        iou = inter / (wh.prod(-1)[:, None] + anc.prod(-1)[None] - inter + 1e-10)
        best = iou.argmax(1)
        for j in range(v):
            g = 2 - best[j] // 3
            r = (32, 16, 8)[g]
            ys[g][i, int(c[j, 1] // r), int(c[j, 0] // r), best[j] % 3, :4] = (c[j, 0], c[j, 1], wh[j, 0], wh[j, 1])
            ys[g][i, int(c[j, 1] // r), int(c[j, 0] // r), best[j] % 3, 4] = 1.0
            ys[g][i, int(c[j, 1] // r), int(c[j, 0] // r), best[j] % 3, 5 + int(rng.integers(0, class_num))] = 1.0
    return [torch.from_numpy(y).cuda() for y in ys]


DUMP_BYTES = 63 * 10**6       # array bytes: the files, .npy headers included, stay under 64 MB


def dump_outputs(path, out, limit=DUMP_BYTES):
    """Write one detection step's results (detect_raw()[1:]: boxes [N,cap,4], scores, labels, indices [N,cap],
    counts [N]) as a caller of detect() receives them: counts.npy and, for every image's first counts[i] slots in
    image order, boxes.npy [K,4], scores.npy [K] (float32), labels.npy and indices.npy [K] (float64, exact).
    When the K rows exceed `limit` bytes in all, a fixed seeded sample of them is written, in order, with their row
    numbers in rows.npy.  Slots past counts[i] are never written by the engine, so they are not dumped."""
    ob, os_, ol, oi, cnt = (t.cpu().numpy() for t in out)
    counts = cnt.astype(np.float64)
    keep = np.arange(ob.shape[1])[None, :] < cnt[:, None]
    arrays = {"boxes": ob[keep], "scores": os_[keep], "labels": ol[keep].astype(np.float64),
              "indices": oi[keep].astype(np.float64)}
    k = len(arrays["scores"])
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    if k * row_bytes + counts.nbytes > limit:
        m = max(0, (limit - counts.nbytes) // (row_bytes + 8))
        rows = np.sort(np.random.default_rng(0).choice(k, size=m, replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    arrays["counts"] = counts
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)
    return sorted(arrays)


# --------------------------------------------------------------------------------------
def latency_b1(pkg, S, iters):
    """Single-image latency (the shape of BASELINE.json configs[0], on the GPU): forward + decode + NMS, one host
    synchronisation per image, CUDA events."""
    import torch
    model = pkg.yolov3(CLASS_NUM, pkg.parse_anchors(os.path.join(ROOT, "yolov3_tensorflow_b200", "data", "yolo_anchors.txt")), dtype="fp16")
    model.init_params(3)
    x = torch.rand((1, S, S, 3), device="cuda")
    ts = []
    for i in range(iters + 5):
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record()
        out = model.detect_raw(x, max_boxes=200, score_thresh=0.3, nms_thresh=0.45)
        b.record(); torch.cuda.synchronize()
        if i >= 5:
            ts.append(a.elapsed_time(b))
    ts.sort()
    tg = []
    for i in range(iters + 5):                  # the same step replayed from a CUDA graph (model.detect_graphed)
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record()
        out = model.detect_graphed(x, max_boxes=200, score_thresh=0.3, nms_thresh=0.45)
        b.record(); torch.cuda.synchronize()
        if i >= 5:
            tg.append(a.elapsed_time(b))
    tg.sort()
    return {"ms_median": ts[len(ts) // 2], "ms_min": ts[0], "images_per_s": 1e3 / ts[len(ts) // 2],
            "cuda_graph_ms_median": tg[len(tg) // 2], "cuda_graph_ms_min": tg[0],
            "what": "batch 1, %dx%d, forward + decode + NMS (yb_net_detect), device-resident input, 76 launches" % (S, S)}


def main():
    sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree (it may be read-only)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=416)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-worker", default=None, help=argparse.SUPPRESS)   # internal: size,steps,warmup,images,threads
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-train608", action="store_true")
    ap.add_argument("--train-batch", type=int, default=32)
    ap.add_argument("--train-size", type=int, default=416)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the detections of the last timed step to DIR/<name>.npy (float32 / float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    workload = (f"batch={args.batch} {args.size}x{args.size} inference: forward + decode + per-image gpu_nms(200, 0.3, 0.45), "
                f"COCO 80-class, random-init cfg-2 weights (BASELINE.json configs[1])")
    config = {"workload": workload, "batch_per_gpu": args.batch, "image": [args.size, args.size], "classes": CLASS_NUM,
              "parallelism": f"replicas x{world} (independent images, no data-path collective)",
              "l2": "per-step inputs (133 MB) + activations (~6 GB) exceed the 126 MB L2; no explicit flush"}

    if args.cpu_worker:
        size, passes, warmup, images, threads = (int(v) for v in args.cpu_worker.split(","))
        print(json.dumps({"pass_seconds": _cpu_worker(size, passes, warmup, images, threads)}))
        return
    if args.impl == "reference":
        if rank != 0:
            return
        steps = args.steps                         # a step = one pass of every worker over its bounded sample
        cb, spp = run_cpu(args.size, steps, 1)
        line = {"impl": "reference", "metric": "images/sec", "value": cb["value"], "unit": "images/s", "n_gpus": args.gpus,
                "steps": steps, "warmup": 1, "ms_per_step": spp * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": cb,
                "product_modules_loaded": sorted(m for m in sys.modules if m.startswith("yolov3_tensorflow_b200")),
                "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    import yolov3_tensorflow_b200 as pkg
    from yolov3_tensorflow_b200 import _lib
    from yolov3_tensorflow_b200.utils.nms_utils import batched_nms_raw

    B, S = args.batch, args.size
    anchors = pkg.parse_anchors(os.path.join(ROOT, "yolov3_tensorflow_b200", "data", "yolo_anchors.txt"))
    model = pkg.yolov3(CLASS_NUM, anchors, dtype="fp16")
    model.set_params(make_bench_params(specs=pkg.yolov3.conv_table(CLASS_NUM)), "HWIO")
    x_host = torch.from_numpy(np.random.default_rng(2 + rank).random((B, S, S, 3), dtype=np.float32)).pin_memory()
    x_dev = x_host.cuda()

    def step_device():
        # forward -> decode -> score -> per-image NMS in one engine call (decode + score filter fused into the
        # detection-head epilogues; bit-identical to forward() + predict_scores() + batched_nms_raw(), tests/test_gpu_path.py)
        return model.detect_raw(x_dev, **NMS_ARGS)[1:]

    def step_device_unfused():
        fms = model.forward(x_dev)
        boxes, scores = model.predict_scores(fms)
        return batched_nms_raw(boxes, scores, CLASS_NUM, **NMS_ARGS)

    # End-to-end pipeline through the public API: pinned host images -> H2D on a copy stream (double buffered,
    # overlapping the previous batch's compute) -> forward/predict/nms -> D2H of the detections into pinned host
    # buffers.  Every step's H2D copy and D2H read happen inside the timed region.
    copy_stream = torch.cuda.Stream()
    x_bufs = [torch.empty_like(x_dev) for _ in range(2)]
    h2d_done = [torch.cuda.Event() for _ in range(2)]
    buf_free = [torch.cuda.Event() for _ in range(2)]
    cap = CLASS_NUM * NMS_ARGS["max_boxes"]
    # detections go back through a D2H stream into double-buffered pinned memory: step i's read-back overlaps step i+1's
    # compute, like the H2D prefetch; the host waits for step i-1's results at the end of step i (and for the last one
    # before the timed region closes), so every step's detections ARE on the host inside the timed region
    d2h_stream = torch.cuda.Stream()
    h_counts = [torch.empty((B,), dtype=torch.int32).pin_memory() for _ in range(2)]
    h_boxes = [torch.empty((B, cap, 4), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_scores = [torch.empty((B, cap), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_labels = [torch.empty((B, cap), dtype=torch.int32).pin_memory() for _ in range(2)]
    d2h_done = [torch.cuda.Event() for _ in range(2)]
    out_keep = [None, None]

    def e2e_prefetch(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(buf_free[i % 2])
            x_bufs[i % 2].copy_(x_host, non_blocking=True)                     # H2D, every step
            h2d_done[i % 2].record(copy_stream)

    def step_e2e(i):
        e2e_prefetch(i + 1)                                                    # next batch's copy overlaps this compute
        cur = torch.cuda.current_stream()
        cur.wait_event(h2d_done[i % 2])
        _, ob, os_, ol, oi, cnt = model.detect_raw(x_bufs[i % 2], **NMS_ARGS)
        buf_free[i % 2].record(cur)
        out_keep[i % 2] = (ob, os_, ol, cnt)                                   # keep the device tensors alive until copied
        computed = torch.cuda.Event(); computed.record(cur)
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(computed)
            h_counts[i % 2].copy_(cnt, non_blocking=True)                      # D2H: K per image
            h_boxes[i % 2].copy_(ob, non_blocking=True)                        # D2H: detections (fixed-size, contiguous)
            h_scores[i % 2].copy_(os_, non_blocking=True)
            h_labels[i % 2].copy_(ol, non_blocking=True)
            d2h_done[i % 2].record(d2h_stream)
        d2h_done[(i - 1) % 2].synchronize()                                    # the PREVIOUS step's results are on the host
        return h_counts[i % 2], cap

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- warm-up ----------------
    for _ in range(max(args.warmup, 3)):
        out = step_device()
    torch.cuda.synchronize()
    n_det = int(out[4].sum())

    # ---------------- timed: device-resident ----------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        last = step_device()
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)

    # ---------------- timed: end to end (host -> host) ----------------
    for ev in buf_free:
        ev.record()
    for ev in d2h_done:
        ev.record()
    e2e_prefetch(0)
    for i in range(2):
        step_e2e(i)
    barrier()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    d2h = 0
    for i in range(2, 2 + args.steps):
        counts, kmax = step_e2e(i)
        d2h = counts.numel() * 4 + B * kmax * (16 + 4 + 4)
    d2h_stream.synchronize()                                                   # the last step's results too
    torch.cuda.current_stream().wait_stream(d2h_stream)
    t1.record()
    barrier()
    ms2 = torch.tensor([t0.elapsed_time(t1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_ms = float(ms2)

    # ---------------- roofline: the tensor-core conv kernel, event-timed inside the step ----------------
    # the same step, its three parts bracketed by events: stem | 74 tcgen05 convs (decode fused into the heads) | NMS
    conv_ms, stem_ms, nms_ms = [], [], []
    res = model.detect_raw(x_dev, **NMS_ARGS)
    for i in range(args.steps + 2):
        a, b, c, d_ = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        a.record()
        model.detect_raw(x_dev, **NMS_ARGS, phases=1, out=res)
        b.record()
        model.detect_raw(x_dev, **NMS_ARGS, phases=2, out=res)
        c.record()
        model.detect_raw(x_dev, **NMS_ARGS, phases=4, out=res)
        d_.record()
        torch.cuda.synchronize()
        if i >= 2:
            stem_ms.append(a.elapsed_time(b)); conv_ms.append(b.elapsed_time(c)); nms_ms.append(c.elapsed_time(d_))
    conv_t = float(np.mean(conv_ms)) * 1e-3
    # the reference-shaped three-call pipeline (forward -> predict -> gpu_nms with fp32 feature maps and scores in HBM)
    for _ in range(3):
        step_device_unfused()
    u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    u0.record()
    for _ in range(args.steps):
        step_device_unfused()
    u1.record()
    torch.cuda.synchronize()
    unfused_ms = u0.elapsed_time(u1) / args.steps
    scale = (S / 416.0) ** 2
    conv_flop = FWD_GFLOP_416 * scale * 1e9 * B          # all 75 convs: the stem runs inside the first tensor-core launch
    pk = peaks()
    achieved = conv_flop / conv_t / 1e12
    traffic = None      # DRAM bytes of the same 74 launches, from the committed ncu table (profiles/, not measured here)
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "conv_traffic.json")))
        if tj.get("batch") == B and tj.get("size") == S:
            traffic = tj["dram_bytes_per_step"]
    except Exception:
        pass
    roofline = {"bound": "tensor", "kernel": "tcgen05 conv kernels (74 launches per step: conv_halo with the stem fused in for layer 1, conv_halo / conv_igemm 1-CTA and CTA-pair kernels for layers 2..74)",
                "achieved": achieved,
                "peak": pk["tflops"], "unit": "TFLOP/s", "frac": achieved / pk["tflops"], "traffic": traffic,
                "peak_source": pk["src"], "ms_per_step_conv": conv_t * 1e3, "ms_per_step_stem": float(np.mean(stem_ms)),
                "ms_per_step_nms": float(np.mean(nms_ms)),
                "algorithmic_flop_per_step": conv_flop}

    # ---------------- training steps (BASELINE.json configs[3] shape: batch 32/GPU @416 bf16; configs[2]: batch 32 @608) ----------------
    train = train608 = None
    if not args.no_train:
        del model, x_dev
        torch.cuda.empty_cache()

        bucket_mb = float(os.environ.get("YB_BUCKET_MB", "32"))     # gradient all-reduce bucket size (0: one blocking all-reduce)

        def bench_train(tb, ts, tsteps):
            tm = pkg.yolov3(CLASS_NUM, anchors, use_label_smooth=True, use_focal_loss=True, batch_norm_decay=0.99, dtype="bf16")
            tm.init_params(seed=3)
            rng = np.random.default_rng(3 + rank)
            xt = torch.from_numpy(rng.random((tb, ts, ts, 3), dtype=np.float32)).cuda()
            yts = synth_y_true(rng, tb, ts, anchors)
            for _ in range(3):
                tm.train_step(xt, yts, 1e-4, bucket_mb=bucket_mb)
            barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(tsteps):
                tl = tm.train_step(xt, yts, 1e-4, bucket_mb=bucket_mb)
            a1.record()
            barrier()
            tms = torch.tensor([a0.elapsed_time(a1)], device="cuda")
            if world > 1:
                dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            t_step = float(tms) / tsteps * 1e-3
            # end to end: pinned host images + ground-truth LISTS -> H2D (copy stream, double buffered) -> y_true built on
            # the device (yb_process_box) -> train step -> D2H of the 5 losses, every step inside the timed region
            from yolov3_tensorflow_b200.utils import data_utils as DU
            bl, ll = synth_gt_lists(np.random.default_rng(30 + rank), tb, ts, CLASS_NUM, 50)
            hb, hl, hc = DU.pack_gt(bl, ll, 50)
            x_h = xt.cpu().pin_memory()
            cs = torch.cuda.Stream()
            xb = [torch.empty_like(xt) for _ in range(2)]
            gb = [(torch.empty_like(hb, device="cuda"), torch.empty_like(hl, device="cuda"), torch.empty_like(hc, device="cuda")) for _ in range(2)]
            yb_ = [[torch.empty_like(y) for y in yts] for _ in range(2)]
            done = [torch.cuda.Event() for _ in range(2)]
            free = [torch.cuda.Event() for _ in range(2)]
            h_loss = torch.empty(5, dtype=torch.float32).pin_memory()

            def prefetch(i):
                with torch.cuda.stream(cs):
                    cs.wait_event(free[i % 2])
                    xb[i % 2].copy_(x_h, non_blocking=True)
                    for d_, h_ in zip(gb[i % 2], (hb, hl, hc)):
                        d_.copy_(h_, non_blocking=True)
                    done[i % 2].record(cs)

            def step_train_e2e(i):
                prefetch(i + 1)
                cur = torch.cuda.current_stream()
                cur.wait_event(done[i % 2])
                y3 = DU.process_box_batch(*gb[i % 2], [ts, ts], CLASS_NUM, anchors, out=yb_[i % 2])
                ls = tm.train_step(xb[i % 2], y3, 1e-4, bucket_mb=bucket_mb)
                free[i % 2].record(cur)
                h_loss.copy_(torch.stack(ls), non_blocking=True)
                cur.synchronize()

            for ev in free:
                ev.record()
            prefetch(0)
            for i in range(2):
                step_train_e2e(i)
            barrier()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            for i in range(2, 2 + tsteps):
                step_train_e2e(i)
            b1.record()
            barrier()
            tme = torch.tensor([b0.elapsed_time(b1)], device="cuda")
            if world > 1:
                dist.all_reduce(tme, op=dist.ReduceOp.MAX)
            e2e_step = float(tme) / tsteps * 1e-3
            gflop = 197.29 * (ts / 416.0) ** 2               # fwd + dgrad + wgrad per image (BASELINE.md §2)
            tfl = tb * gflop * 1e9 / t_step / 1e12
            out = {"images_per_s": tb * world / t_step, "ms_per_step": t_step * 1e3, "batch_per_gpu": tb, "image": [ts, ts],
                   "dtype": "bf16", "loss_total": float(tl[0]), "steps": tsteps, "warmup": 3,
                   "e2e": {"value": tb * world / e2e_step, "unit": "images/s", "ms_per_step": e2e_step * 1e3,
                           "h2d_bytes_per_step": int(x_h.numel() * 4 + hb.numel() * 4 + hl.numel() * 4 + hc.numel() * 4),
                           "d2h_bytes_per_step": 20,
                           "what": "pinned host images + gt box lists -> H2D -> y_true on the device (yb_process_box) -> train step -> losses to the host"},
                   "roofline": {"bound": "tensor", "kernel": "whole training step (conv fwd + dgrad + wgrad FLOPs / step time)",
                                "achieved": tfl, "peak": pk["tflops"], "unit": "TFLOP/s", "frac": tfl / pk["tflops"],
                                "algorithmic_flop_per_step": tb * gflop * 1e9, "peak_source": pk["src"]},
                   "tflops": tfl, "frac_of_peak": tfl / pk["tflops"],
                   "what": "forward(BN batch stats) + compute_loss(focal, label-smooth) + backward + "
                           + (("NCCL all-reduce in %g MB buckets overlapping the backward + " % bucket_mb if bucket_mb > 0 else "one blocking NCCL all-reduce + ") if world > 1 else "")
                           + "L2/clip/momentum update, synthetic <=50 boxes/img"}
            del tm, xt, yts, xb, gb, yb_
            torch.cuda.empty_cache()
            return out

        train = bench_train(args.train_batch, args.train_size, args.steps)
        train["config"] = "BASELINE.json configs[3] per-GPU shape: batch %d x %d GPU(s), 416x416, bf16, data-parallel" % (args.train_batch, world)
        if world == 1 and not args.no_train608:
            train608 = bench_train(32, 608, args.steps)
            train608["config"] = "BASELINE.json configs[2]: batch=32 608x608 training step, random init, 1 GPU"

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    imgs = B * world * args.steps
    value = imgs / (ms_total * 1e-3)
    line = {"metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic", "config": config,
            "e2e": {"value": imgs / (e2e_ms * 1e-3), "unit": "images/s", "h2d_bytes_per_step": x_host.numel() * 4,
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": args.steps * (74 + 2),
            "launches_per_step": {"stem (mma.sync) fused into Conv_1's halo producer + conv_halo / conv_igemm (tcgen05: halo-tile, 1-CTA, CTA-pair kernels; decode + score filter in the 3 head epilogues)": 74,
                                  "nms_select + nms_gather": 2},
            "unfused_api_ms_per_step": unfused_ms,
            "detections_per_step": n_det, "clocks": clocks, "roofline": roofline,
            "fraction_of_conv_flop_roofline": (value / world) * FWD_GFLOP_416 * scale * 1e9 / (pk["tflops"] * 1e12)}
    if train is not None:
        line["train"] = train
    if train608 is not None:
        line["train608"] = train608
    if world == 1:
        line["latency_batch1"] = latency_b1(pkg, S, args.steps)
    if world == 1:
        line["nms_stress"] = nms_stress(pkg, with_cpu=not args.no_cpu_baseline, iters=args.steps)
    if world == 1 and not args.no_cpu_baseline:
        cb, _ = run_cpu(S, 3, 1)
        line["cpu_baseline"] = cb
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
