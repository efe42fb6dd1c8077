"""The matching stage on dense prompt grids: 4 096, 8 192 and 16 384 candidate masks per image (points_per_side 64,
90 and 128).

    python tools/dense_grid_throughput.py [--sizes 4096 8192 16384] [--sets 16] [--streams 16] [--rounds 24]
                                          [--reps 3] [--out profiles/dense_grid_throughput.json]

Config-2 shapes otherwise (ViT-L features C = 1024, 80 classes, 1024 x 1024 output, top-100).  Per size:

  throughput    `--sets` resident single-plane input sets generated on the device (4 GB of logits each at 16 384
                masks, far beyond the 126 MB of L2), consumed in rotation, image i on stream slot i % streams, one bound
                graph per slot (`graphed(..., bind=True)`, each replay binding the set's own tensors); CUDA events on the
                launching stream around `--rounds` passes over all sets after two warm-up passes; median of `--reps`.
  latency       one image at a time in low-latency mode (bound graph replay, then synchronise), median of `--reps`
                runs of `--ll-images` images; and the per-stage split of eager low-latency calls
                (`stage.profile(True)` / `profile_read()`, CUDA events between the stages, median over the images).
  kernels       CUDA time per image of the NMS and pooling-order kernels (`torch.profiler`, a separate run of eager
                throughput-mode calls): the single-CTA score sort (which also clears the `nz` summary of n * n / 1024
                words), the single-CTA class-order sort, the suppression matrix and the scan.
  HBM floor     4 * n * 65 536 bytes of logits at the copy peak measured in the same run (a device-to-device copy of
                8 GB), over the measured time per image.

Before timing, every set's bound-graph result is compared with the eager result (counts, scores with their NaN
pattern, labels, boxes, index, masks).  The card's name, power limit and max SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FEAT, N_CLS, NUM_OUT = 1024, 80, 100
HW = (1024, 1024)
PLANE = 256 * 256


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else ""
    return dict(name=torch.cuda.get_device_name(), nvidia_smi_name_power_limit_max_sm_clock=line)


def copy_peak_gbs(dev, nbytes=8 << 30, reps=5):
    """Device-to-device copy rate (bytes read + written per second), best of `reps`."""
    a = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    best = 0.0
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        best = max(best, 2 * nbytes / (e0.elapsed_time(e1) / 1e3) / 1e9)
    del a, b
    torch.cuda.empty_cache()
    return best


def same(a, b):
    return (a["counts"] == b["counts"] and torch.equal(torch.isnan(a["scores"]), torch.isnan(b["scores"]))
            and torch.equal(torch.nan_to_num(a["scores"]), torch.nan_to_num(b["scores"]))
            and torch.equal(a["labels"], b["labels"]) and torch.equal(a["bboxes"], b["bboxes"])
            and torch.equal(a["index"], b["index"]) and torch.equal(a["binary_masks"], b["binary_masks"]))


KERNELS = ("nms_sort_kernel", "nms_class_sort_kernel", "nms_mask_kernel", "nms_wave_sparse_kernel", "nms_wave_kernel",
           "pool_order_kernel")


def kernel_us(stage, sets, images, dev):
    """CUDA microseconds per image of the kernels named in KERNELS (eager throughput-mode calls under torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    for i in range(4):
        stage.match_async(*sets[i % len(sets)], HW, slot="prof").get()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(images):
            stage.match_async(*sets[i % len(sets)], HW, slot="prof")
        torch.cuda.synchronize(dev)
    out = {}
    for ev in prof.key_averages():
        if any(k in ev.key for k in KERNELS):
            name = ev.key.split("(")[0].replace("void ", "").replace("nttt::", "")  # (template arguments kept)
            t = getattr(ev, "device_time_total", None)
            out[name] = out.get(name, 0.0) + (t if t is not None else ev.cuda_time_total) / images
    return out


def one_size(pkg, stage, n, args, dev, centres, peak_gbs):
    synth = pkg.synth
    S, K = args.streams, args.sets
    streams = [torch.cuda.Stream(dev) for _ in range(S)]
    sets = [synth.make_stage_inputs_device(n, centres, dev, seed=1234 + i) for i in range(K)]
    torch.cuda.synchronize()
    outs = [(torch.zeros((NUM_OUT, *HW), dtype=torch.uint8, device=dev),
             torch.zeros((NUM_OUT, 4), dtype=torch.int32, device=dev)) for _ in range(S)]
    graphs = [stage.graphed(n, FEAT, HW, key=("dense", n, s), persistent_out=outs[s], bind=True).capture()
              for s in range(S)]

    def replay(g, i):
        lr, ious, feat = sets[i]
        return g.replay(lr_masks=lr, pred_ious=ious, tar_feat=feat)

    bad = [i for i in range(K) if not same(replay(graphs[i % S], i).get(),
                                           stage.match_async(*sets[i], HW, slot="check").get())]

    def step():
        for i in range(K):
            with torch.cuda.stream(streams[i % S]):
                replay(graphs[i % S], i)

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    runs = []
    for _ in range(args.reps):
        cur = torch.cuda.current_stream(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(cur)
        for s in streams:
            s.wait_event(e0)
        for _ in range(args.rounds):
            step()
        for s in streams:
            cur.wait_stream(s)
        e1.record(cur)
        torch.cuda.synchronize()
        runs.append(1e3 * e0.elapsed_time(e1) / (args.rounds * K))
    us = statistics.median(runs)
    floor_us = 4 * n * PLANE / (peak_gbs * 1e9) * 1e6
    del graphs, outs
    torch.cuda.synchronize()

    # ---- one image at a time, low-latency launch shapes
    g_ll = stage.graphed(n, FEAT, HW, key=("dense_ll", n), low_latency=True, bind=True).capture()
    ll_bad = [i for i in range(min(K, 4)) if not same(replay(g_ll, i).get(), stage.match(*sets[i], HW, low_latency=True))]
    for i in range(10):
        replay(g_ll, i % K)
    torch.cuda.synchronize()
    ll_runs = []
    for _ in range(args.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.ll_images):
            replay(g_ll, i % K)
            torch.cuda.current_stream().synchronize()
        e1.record()
        torch.cuda.synchronize()
        ll_runs.append(1e3 * e0.elapsed_time(e1) / args.ll_images)
    del g_ll
    stage.profile(True)
    per_stage = {}
    for i in range(args.ll_images):
        stage.match(*sets[i % K], HW, low_latency=True)
        for k, v in stage.profile_read().items():
            per_stage.setdefault(k, []).append(1e3 * v)
    stage.profile(False)
    split = {k: statistics.median(v) for k, v in per_stage.items()}
    kern = kernel_us(stage, sets, args.prof_images, dev)
    del sets
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return dict(masks=n, points_per_side=round(n ** 0.5, 1),
                throughput=dict(us_per_image=us, images_per_s=1e6 / us, runs_us=runs),
                hbm_floor=dict(logits_bytes=4 * n * PLANE, floor_us=floor_us, frac_of_floor=floor_us / us),
                low_latency_one_image=dict(us_per_image=statistics.median(ll_runs), runs_us=ll_runs,
                                           per_stage_us=split),
                kernel_us_per_image=kern,
                outputs_equal_eager=dict(sets=K, mismatches=bad, low_latency_mismatches=ll_bad))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[4096, 8192, 16384])
    ap.add_argument("--sets", type=int, default=16)
    ap.add_argument("--streams", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=24, help="timed passes over all sets per measurement")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ll-images", type=int, default=50, help="images per low-latency measurement")
    ap.add_argument("--prof-images", type=int, default=8, help="images under torch.profiler per size")
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device (there is no CPU path)"
    pkg = importlib.import_module("no-time-to-train_b200")
    dev = torch.device("cuda", 0)
    centres = pkg.synth.cluster_centres(FEAT)
    gen = torch.Generator().manual_seed(args.seed)
    protos = centres[torch.arange(N_CLS) % centres.shape[0]] + 0.05 * torch.randn(N_CLS, FEAT, generator=gen)
    stage = pkg.MatchingStage(dev, pkg.StageConfig(nms_thr=0.5, num_out_instance=NUM_OUT, enc_hw=(37, 37)))
    stage.set_prototypes(protos.unsqueeze(1))
    peak = copy_peak_gbs(dev)
    sizes = [one_size(pkg, stage, n, args, dev, centres, peak) for n in args.sizes]
    rec = dict(tool="tools/dense_grid_throughput.py", card=card(), copy_peak_gbs=peak, resident_sets=args.sets,
               streams=args.streams, rounds=args.rounds, reps=args.reps, feat_dim=FEAT, classes=N_CLS,
               num_out_instance=NUM_OUT, out_hw=HW, sizes=sizes,
               timing="CUDA events; throughput: bound graphs per stream slot over resident sets in HBM; latency: "
                      "low-latency bound graph replay + synchronise per image; per-stage split: profile events of "
                      "eager low-latency calls; kernels: torch.profiler in a separate pass")
    print(json.dumps(rec))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")
    bad = {s["masks"]: s["outputs_equal_eager"] for s in sizes
           if s["outputs_equal_eager"]["mismatches"] or s["outputs_equal_eager"]["low_latency_mismatches"]}
    if bad:
        raise SystemExit(f"bound-graph outputs differ from the eager stage: {bad}")


if __name__ == "__main__":
    main()
