"""Throughput of the matching stage on compacted candidate lists (the reference's `masks[keep]` after
`scores > iou_thr`), whose length changes from image to image.

    python tools/candidate_count_throughput.py [--sets 32] [--streams 16] [--rounds 10] [--reps 3] [--out F]

Config-2 shapes (ViT-L features C = 1024, 80 classes, 1024 x 1024 output, iou_thr 0.5), single-plane inputs generated
on the device.  `--sets` resident input sets of 4096 candidates each; set i has its own count, drawn with a fixed seed
from [512, 1024] for capacity 1024 and from [2048, 4096] for capacity 4096 (its first k rows are the compacted list).
Image i runs on stream slot i % streams with graphs held per stream slot.  In microseconds per image (CUDA events on
the launching stream around `--rounds` passes over all sets, after two warm-up passes; the modes alternate in one
session, `--reps` times each, median reported):

  (a) eager_<cap>        `match_async` on the k-row tensors (nttt_match_image at k);
  (b) padded_<cap>       a static graph at the capacity: `copy_` of the k rows into its buffers and NaN IoUs past k, so
                         that the fused filter drops them (the best a graph user can do without the counted entry);
  (c) counted_<cap>      a bound, counted graph at the capacity (`graphed(cap, ..., bind=True, counted=True)`) replayed
                         on the k-row tensors;
  (d) counted_1024_full / bound_1024_full: every set's first 1024 rows, the counted graph at its capacity against a
                         bound graph captured at n = 1024;
  (e) counted_4096_at_1024 / bound_1024_full: the capacity-4096 counted graph serving the same 1024 rows;
  (f) one image at a time in low-latency mode (replay, then synchronise): a counted graph of capacity 1024 at k = 1000
      against a bound graph captured at 1000.

Before timing, every mode's outputs for every set are compared with the eager stage on the k-row tensors: counts, scores
(NaN pattern included), labels, boxes, index and masks must be identical.  The card's name, power limit and max SM
clock are read in the same run.
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

FEAT, N_CLS, SHOTS, THR = 1024, 80, 10, 0.5
HW = (1024, 1024)
CAPS = {1024: (512, 1024), 4096: (2048, 4096)}
LL_K = 1000


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else ""
    return dict(name=torch.cuda.get_device_name(), nvidia_smi=line)


def same(a, b):
    return (a["counts"] == b["counts"] and torch.equal(torch.isnan(a["scores"]), torch.isnan(b["scores"]))
            and torch.equal(torch.nan_to_num(a["scores"]), torch.nan_to_num(b["scores"]))
            and torch.equal(a["labels"], b["labels"]) and torch.equal(a["bboxes"], b["bboxes"])
            and torch.equal(a["index"], b["index"]) and torch.equal(a["binary_masks"], b["binary_masks"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sets", type=int, default=32)
    ap.add_argument("--streams", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=10, help="timed passes over all sets per measurement")
    ap.add_argument("--reps", type=int, default=3, help="alternating repetitions of each mode")
    ap.add_argument("--ll-images", type=int, default=200, help="images per low-latency measurement")
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device (there is no CPU path)"
    pkg = importlib.import_module("no-time-to-train_b200")
    dev = torch.device("cuda", 0)
    synth = pkg.synth
    centres = synth.cluster_centres(FEAT)
    stage = pkg.MatchingStage(dev, pkg.StageConfig(nms_thr=0.5, num_out_instance=100, enc_hw=(37, 37)))
    gen = torch.Generator().manual_seed(args.seed)
    stage.set_prototypes(centres[torch.arange(N_CLS) % centres.shape[0]].unsqueeze(1)
                         + 0.05 * torch.randn(N_CLS, SHOTS, FEAT, generator=gen))
    S, K = args.streams, args.sets
    streams = [torch.cuda.Stream(dev) for _ in range(S)]
    num_out = stage.cfg.num_out_instance
    sets = [synth.make_stage_inputs_device(max(CAPS), centres, dev, seed=1234 + i) for i in range(K)]
    counts = {cap: torch.randint(lo, hi + 1, (K,), generator=gen).tolist() for cap, (lo, hi) in CAPS.items()}
    torch.cuda.synchronize()

    def rows(i, k):
        lr, ious, feat = sets[i]
        return lr[:k], ious[:k], feat

    def graphs(tag, n, **kw):
        gs = []
        for s in range(S):
            out = (torch.zeros((num_out, *HW), dtype=torch.uint8, device=dev),
                   torch.zeros((num_out, 4), dtype=torch.int32, device=dev))
            gs.append(stage.graphed(n, FEAT, HW, iou_thr=THR, key=(tag, s), persistent_out=out, **kw).capture())
        return gs

    def eager(cap):
        return lambda i: stage.match_async(*rows(i, counts[cap][i]), HW, iou_thr=THR, slot=("eager", i % S))

    def padded(gs, cap):
        def fn(i):
            g, k = gs[i % S], counts[cap][i]
            lr, ious, feat = sets[i]
            g.lr_masks[:k].copy_(lr[:k])
            g.pred_ious[:k].copy_(ious[:k])
            g.pred_ious[k:].fill_(float("nan"))
            g.tar_feat.copy_(feat)
            return g.replay()
        return fn

    def counted(gs, cap):
        def fn(i):
            lr, ious, feat = rows(i, counts[cap][i])
            return gs[i % S].replay(lr_masks=lr, pred_ious=ious, tar_feat=feat)
        return fn

    def full(gs):
        def fn(i):
            lr, ious, feat = rows(i, 1024)
            return gs[i % S].replay(lr_masks=lr, pred_ious=ious, tar_feat=feat)
        return fn

    g_pad = {cap: graphs(f"padded_{cap}", cap) for cap in CAPS}
    g_cnt = {cap: graphs(f"counted_{cap}", cap, bind=True, counted=True) for cap in CAPS}
    g_b1024 = graphs("bound_1024", 1024, bind=True)
    modes = {}
    for cap in CAPS:
        modes[f"eager_{cap}"] = (eager(cap), cap)
        modes[f"padded_{cap}"] = (padded(g_pad[cap], cap), cap)
        modes[f"counted_{cap}"] = (counted(g_cnt[cap], cap), cap)
    modes["counted_1024_full"] = (full(g_cnt[1024]), None)
    modes["bound_1024_full"] = (full(g_b1024), None)
    modes["counted_4096_at_1024"] = (full(g_cnt[4096]), None)
    # ---- outputs == eager at k, for every set and mode
    bad = []
    for i in range(K):
        refs = {cap: stage.match_async(*rows(i, counts[cap][i]), HW, iou_thr=THR, slot="check").get() for cap in CAPS}
        ref_full = stage.match_async(*rows(i, 1024), HW, iou_thr=THR, slot="check").get()
        for name, (fn, cap) in modes.items():
            if not name.startswith("eager") and not same(fn(i).get(), refs[cap] if cap else ref_full):
                bad.append((i, name))

    def on_streams(fn):
        def step():
            for i in range(K):
                with torch.cuda.stream(streams[i % S]):
                    fn(i)
        return step

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
        return 1e3 * e0.elapsed_time(e1) / (args.rounds * K)

    steps = {name: on_streams(fn) for name, (fn, _) in modes.items()}
    for step in steps.values():
        for _ in range(2):
            step()
    torch.cuda.synchronize()
    got = {k: [] for k in steps}
    for _ in range(args.reps):
        for k, step in steps.items():
            got[k].append(timed(step))
    res = {k: dict(us_per_image=statistics.median(v), runs=v) for k, v in got.items()}
    del g_pad, g_cnt, g_b1024
    torch.cuda.synchronize()

    # ---- (f) one image at a time, low-latency launch shapes
    def one(tag, n, **kw):
        out = (torch.zeros((num_out, *HW), dtype=torch.uint8, device=dev),
               torch.zeros((num_out, 4), dtype=torch.int32, device=dev))
        return stage.graphed(n, FEAT, HW, iou_thr=THR, key=tag, persistent_out=out, low_latency=True, **kw).capture()

    g_ll = {"counted_1024_at_1000": one("ll_counted", 1024, bind=True, counted=True),
            "bound_1000": one("ll_bound", LL_K, bind=True)}

    def ll(g):
        def fn(i):
            lr, ious, feat = rows(i % K, LL_K)
            return g.replay(lr_masks=lr, pred_ious=ious, tar_feat=feat)
        return fn

    ll_modes = {k: ll(g) for k, g in g_ll.items()}
    ll_bad = [(i, k) for i in range(K) for k, fn in ll_modes.items()
              if not same(fn(i).get(), stage.match_async(*rows(i, LL_K), HW, iou_thr=THR, slot="ll",
                                                         low_latency=True).get())]
    lat = {k: [] for k in ll_modes}
    for fn in ll_modes.values():
        for i in range(10):
            fn(i)
    torch.cuda.synchronize()
    for _ in range(args.reps):
        for k, fn in ll_modes.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.ll_images):
                fn(i)
                torch.cuda.current_stream().synchronize()
            e1.record()
            torch.cuda.synchronize()
            lat[k].append(1e3 * e0.elapsed_time(e1) / args.ll_images)
    res_ll = {k: dict(us_per_image=statistics.median(v), runs=v) for k, v in lat.items()}

    rec = dict(tool="tools/candidate_count_throughput.py", card=card(), resident_sets=K, streams=S, rounds=args.rounds,
               reps=args.reps, feat_dim=FEAT, classes=N_CLS, num_out_instance=num_out, out_hw=HW, iou_thr=THR,
               counts={str(cap): dict(range=list(r), mean=statistics.mean(counts[cap])) for cap, r in CAPS.items()},
               outputs_equal_eager=dict(images=K, mismatches=bad, low_latency_mismatches=ll_bad),
               throughput=res, low_latency_one_image=dict(k=LL_K, **res_ll),
               timing="CUDA events on the launching stream; inputs resident in HBM, rotating over the sets; graphs per "
                      "stream slot; modes alternate in one session; median of --reps runs")
    print(json.dumps(rec))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")
    if bad or ll_bad:
        raise SystemExit(f"outputs differ from the eager stage: {bad}, low latency {ll_bad}")


if __name__ == "__main__":
    main()
