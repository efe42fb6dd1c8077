"""Throughput of the matching stage on a dataset of mixed image sizes (COCO-like: long side <= 640).

    python tools/mixed_size_throughput.py [--images 256] [--streams 16] [--rounds 5] [--out FILE.json]

Config-2 shapes (1024 masks, ViT-L features, 80 classes), inputs resident in HBM and generated on the device with the
recipes bench.py uses.  Every image has its own output size from a seeded mix.  Reported, in images/s (CUDA events on
the launching stream around `--rounds` passes over all images, after two warm-up passes; modes alternate in one session,
`--reps` times each, median and spread reported):

  1. sized_graph      one sized CUDA graph per resident image and stream slot (`graphed(..., min_hw=...)`: its tensors
                      are the static inputs, as in bench.py), each replayed at its image's size;
  2. eager            `match_async` in throughput mode on the same streams, each call at its image's size;
  3. at_1024          every image at 1024 x 1024: the sized graph (capacity 1024^2) against the static graph;
  4. low_latency      one image at a time (replay + synchronise), 1024 x 1024, sized against static, in microseconds.

Before timing, every image's outputs of (1) are compared with (2): counts, scores (NaN pattern included), labels, boxes,
index and masks must be identical.  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import random
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# COCO-like output sizes (h, w): the common 640-long-side shapes and a few others
SIZE_MIX = [(480, 640), (640, 480), (427, 640), (640, 427), (333, 500), (375, 500), (612, 612), (640, 640),
            (500, 375), (424, 640), (640, 512), (360, 480)]
CAP, MIN_HW = (640, 640), (256, 256)
N_MASKS, FEAT, N_CLS = 1024, 1024, 80


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else ""
    return dict(name=torch.cuda.get_device_name(), nvidia_smi=line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=256)
    ap.add_argument("--streams", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=5, help="timed passes over all images per measurement")
    ap.add_argument("--reps", type=int, default=3, help="alternating repetitions of each comparison")
    ap.add_argument("--ll-images", type=int, default=200, help="images per low-latency measurement")
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device (there is no CPU path)"
    pkg = importlib.import_module("no-time-to-train_b200")
    dev = torch.device("cuda", 0)
    synth = pkg.synth
    centres = synth.cluster_centres(FEAT)
    gen = torch.Generator().manual_seed(args.seed)
    protos = (centres[torch.arange(N_CLS) % centres.shape[0]] + 0.05 * torch.randn(N_CLS, FEAT, generator=gen))
    stage = pkg.MatchingStage(dev, pkg.StageConfig(nms_thr=0.5, num_out_instance=100, enc_hw=(37, 37)))
    stage.set_prototypes(protos.unsqueeze(1))
    rng = random.Random(args.seed)
    sizes = [rng.choice(SIZE_MIX) for _ in range(args.images)]
    resident = [synth.make_stage_inputs_device(N_MASKS, centres, dev, seed=1234 + i) for i in range(args.images)]
    S = args.streams
    streams = [torch.cuda.Stream(dev) for _ in range(S)]
    num_out = stage.cfg.num_out_instance

    def outs(hw):
        return [(torch.zeros((num_out, *hw), dtype=torch.uint8, device=dev),
                 torch.zeros((num_out, 4), dtype=torch.int32, device=dev)) for _ in range(S)]

    def graphs(tag, hw, min_hw, low_latency=False, count=None):
        o = outs(hw)
        gs = []
        for i in range(count or args.images):
            g = stage.graphed(N_MASKS, FEAT, hw, key=(tag, i % S), persistent_out=o[i % S], low_latency=low_latency,
                              min_hw=min_hw)
            g.lr_masks, g.pred_ious, g.tar_feat = resident[i]
            gs.append(g.capture())
        return gs

    t0 = time.perf_counter()
    sized = graphs("sized", CAP, MIN_HW)
    capture_s = time.perf_counter() - t0
    atlas_cap640 = stage.atlas_stats()

    # ---- outputs of (1) == (2), image by image
    mism = []
    for i, g in enumerate(sized):
        out = g.replay(ori_hw=sizes[i]).get()
        ref = stage.match_async(*resident[i], sizes[i], slot="check").get()
        same = (out["counts"] == ref["counts"] and torch.equal(torch.isnan(out["scores"]), torch.isnan(ref["scores"]))
                and torch.equal(torch.nan_to_num(out["scores"]), torch.nan_to_num(ref["scores"]))
                and torch.equal(out["labels"], ref["labels"]) and torch.equal(out["bboxes"], ref["bboxes"])
                and torch.equal(out["index"], ref["index"]) and torch.equal(out["binary_masks"], ref["binary_masks"]))
        if not same:
            mism.append(i)
    torch.cuda.synchronize()

    def timed(step):
        cur = torch.cuda.current_stream(dev)
        torch.cuda.synchronize()
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
        return args.rounds * args.images / (e0.elapsed_time(e1) / 1e3)

    def run_graphs(gs, hw_of):
        def step():
            for i, g in enumerate(gs):
                with torch.cuda.stream(streams[i % S]):
                    g.replay(ori_hw=hw_of(i)) if g.min_hw is not None else g.replay()
        return step

    def run_eager(hw_of):
        def step():
            for i in range(args.images):
                with torch.cuda.stream(streams[i % S]):
                    stage.match_async(*resident[i], hw_of(i), slot=("eager", i % S))
        return step

    def compare(modes):
        """modes: name -> step; warm-up twice each, then `reps` alternating rounds"""
        for step in modes.values():
            for _ in range(2):
                step()
        torch.cuda.synchronize()
        got = {k: [] for k in modes}
        for _ in range(args.reps):
            for k, step in modes.items():
                got[k].append(timed(step))
        return {k: dict(images_per_s=statistics.median(v), runs=v) for k, v in got.items()}

    res_mixed = compare({"sized_graph": run_graphs(sized, lambda i: sizes[i]), "eager": run_eager(lambda i: sizes[i])})
    del sized
    torch.cuda.synchronize()
    big = (1024, 1024)
    sized_big = graphs("sized1024", big, MIN_HW)
    static_big = graphs("static1024", big, None)
    atlas_all = stage.atlas_stats()
    res_1024 = compare({"sized_graph": run_graphs(sized_big, lambda i: big),
                        "static_graph": run_graphs(static_big, lambda i: big)})
    del sized_big, static_big
    torch.cuda.synchronize()

    # ---- one image at a time, low-latency launch shapes
    ll = {"sized_graph": graphs("ll_sized", big, MIN_HW, low_latency=True, count=1)[0],
          "static_graph": graphs("ll_static", big, None, low_latency=True, count=1)[0]}
    lat = {k: [] for k in ll}
    for k, g in ll.items():
        for _ in range(10):
            g.replay(ori_hw=big)
        torch.cuda.synchronize()
    for _ in range(args.reps):
        for k, g in ll.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.ll_images):
                g.replay(ori_hw=big)
                torch.cuda.current_stream().synchronize()
            e1.record()
            torch.cuda.synchronize()
            lat[k].append(1e3 * e0.elapsed_time(e1) / args.ll_images)
    res_ll = {k: dict(us_per_image=statistics.median(v), runs=v) for k, v in lat.items()}

    rec = dict(tool="tools/mixed_size_throughput.py", card=card(), images=args.images, streams=S, rounds=args.rounds,
               reps=args.reps, masks=N_MASKS, feat_dim=FEAT, classes=N_CLS, num_out_instance=num_out,
               capacity=CAP, min_hw=MIN_HW, size_mix=SIZE_MIX, sizes_drawn={f"{h}x{w}": sizes.count((h, w))
                                                                              for h, w in SIZE_MIX},
               outputs_sized_equal_eager=dict(images=args.images, mismatches=mism),
               capture_s_sized_graphs=capture_s,
               atlas_640=atlas_cap640, atlas_640_and_1024=atlas_all,
               mixed_sizes=res_mixed, at_1024=res_1024, low_latency_1024=res_ll,
               timing="CUDA events on the launching stream; inputs resident in HBM; modes alternate in one session")
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")
    if mism:
        raise SystemExit(f"outputs of the sized graphs differ from the eager stage on images {mism}")


if __name__ == "__main__":
    main()
