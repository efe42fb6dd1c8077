"""Throughput of the matching stage when the memory bank changes from image to image (a seed / shot sweep, or a server
holding several few-shot tasks).

    python tools/bank_switch_throughput.py [--sets 32] [--streams 16] [--banks 8] [--rounds 20] [--reps 3] [--out F]

Config-2 shapes (1024 masks, ViT-L features C = 1024, 1024 x 1024 output), single-plane inputs generated on the device.
`--sets` resident input sets (268 MB of logits each, far more than the 126 MB of L2 in total) are consumed in rotation,
image i on stream slot i % streams with graphs held per stream slot, and image i is scored against bank
(i + i // streams) % banks: consecutive images, and consecutive replays of one slot's graph, use different banks.  The
banks are `--banks` seeded draws of 80 classes x 10 shots around the same class centres (one bank per seed of a sweep),
prepared once.  In images/s (CUDA events on the launching stream around `--rounds` passes over all sets, after two
warm-up passes; the modes alternate in one session, `--reps` times each):

  eager            `match_async` in throughput mode, the stage's prototypes switched to the image's bank;
  recapture        a bound graph per slot (`graphed(..., bind=True)`), the stage's prototypes switched to the image's
                   bank: the graph re-captures whenever they changed since its capture (every image here);
                   `--recapture-rounds` passes only;
  banked_80        a bound, banked graph per slot (`bank_capacity=(80, 0)`), each replay binding the image's bank;
  banked_1203      the same at a capacity of 1203 classes (LVIS), serving the same 80-class banks.

Also one image at a time in low-latency mode (replay, then synchronise), in microseconds: the banked graph switching
banks every image, and the bound graph on one fixed bank.

Before timing, the outputs of every image of a pass are compared with the eager stage on its bank: counts, scores (NaN
pattern included), labels, boxes, index and masks must be identical for recapture and banked_80, whose launch shapes are
the eager stage's; for banked_1203 the number of identical images is reported.  The card's name and power limit are read
in the same run.
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

N_MASKS, FEAT, N_CLS, SHOTS, LVIS = 1024, 1024, 80, 10, 1203
HW = (1024, 1024)


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
    ap.add_argument("--banks", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=20, help="timed passes over all sets per measurement")
    ap.add_argument("--recapture-rounds", type=int, default=2, help="timed passes of the re-capturing mode")
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
    stage = pkg.MatchingStage(dev, pkg.StageConfig(nms_thr=0.5, num_out_instance=100, enc_hw=(37, 37)))
    banks = []
    for b in range(args.banks):  # the seeds of a sweep: the same classes, other reference shots
        gen = torch.Generator().manual_seed(args.seed + b)
        shots = (centres[torch.arange(N_CLS) % centres.shape[0]].unsqueeze(1)
                 + 0.05 * torch.randn(N_CLS, SHOTS, FEAT, generator=gen))
        banks.append(stage.prepare_bank(shots))
    S, K, B = args.streams, args.sets, args.banks
    streams = [torch.cuda.Stream(dev) for _ in range(S)]
    num_out = stage.cfg.num_out_instance
    single = [synth.make_stage_inputs_device(N_MASKS, centres, dev, seed=1234 + i) for i in range(K)]
    torch.cuda.synchronize()
    stage._use_bank(banks[0])

    def bank_of(i):
        return banks[(i + i // S) % B]

    def per_slot(tag, low_latency=False, count=None, bank_capacity=None):
        gs = []
        for s in range(count or S):
            out = (torch.zeros((num_out, *HW), dtype=torch.uint8, device=dev),
                   torch.zeros((num_out, 4), dtype=torch.int32, device=dev))
            gs.append(stage.graphed(N_MASKS, FEAT, HW, key=(tag, s), persistent_out=out, low_latency=low_latency,
                                    bind=True, bank_capacity=bank_capacity).capture(banks[0]))
        return gs

    def eager(i, slot, low_latency=False):
        stage._use_bank(bank_of(i))
        return stage.match_async(*single[i % K], HW, slot=slot, low_latency=low_latency)

    def recapture(g, i):
        stage._use_bank(bank_of(i))
        lr, ious, feat = single[i % K]
        return g.replay(lr_masks=lr, pred_ious=ious, tar_feat=feat)

    def banked(g, i):
        lr, ious, feat = single[i % K]
        return g.replay(lr_masks=lr, pred_ious=ious, tar_feat=feat, bank=bank_of(i))

    def timed(step, rounds):
        cur = torch.cuda.current_stream(dev)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(cur)
        for s in streams:
            s.wait_event(e0)
        for _ in range(rounds):
            step()
        for s in streams:
            cur.wait_stream(s)
        e1.record(cur)
        torch.cuda.synchronize()
        return rounds * K / (e0.elapsed_time(e1) / 1e3)

    def on_streams(fn):
        def step():
            for i in range(K):
                with torch.cuda.stream(streams[i % S]):
                    fn(i)
        return step

    g_re = per_slot("recapture")
    g_80 = per_slot("banked_80", bank_capacity=(N_CLS, 0))
    g_1203 = per_slot("banked_1203", bank_capacity=(LVIS, 0))
    # ---- outputs == eager on the image's bank, for every image of a pass (set, bank and slot as the timed passes)
    bad, identical_1203 = [], 0
    for i in range(K):
        ref = eager(i, "check").get()
        if not same(recapture(g_re[i % S], i).get(), ref):
            bad.append((i, "recapture"))
        if not same(banked(g_80[i % S], i).get(), ref):
            bad.append((i, "banked_80"))
        identical_1203 += same(banked(g_1203[i % S], i).get(), ref)
    modes = {"eager": (on_streams(lambda i: eager(i, ("eager", i % S))), args.rounds),
             "recapture": (on_streams(lambda i: recapture(g_re[i % S], i)), args.recapture_rounds),
             "banked_80": (on_streams(lambda i: banked(g_80[i % S], i)), args.rounds),
             "banked_1203": (on_streams(lambda i: banked(g_1203[i % S], i)), args.rounds)}
    for step, _ in modes.values():
        for _ in range(2):
            step()
    torch.cuda.synchronize()
    got = {k: [] for k in modes}
    for _ in range(args.reps):
        for k, (step, rounds) in modes.items():
            got[k].append(timed(step, rounds))
    res = {k: dict(images_per_s=statistics.median(v), us_per_image=1e6 / statistics.median(v), runs=v)
           for k, v in got.items()}
    del g_re, g_80, g_1203
    torch.cuda.synchronize()

    # ---- one image at a time, low-latency launch shapes
    stage._use_bank(banks[0])
    g_bound = per_slot("ll_bound", low_latency=True, count=1)[0]
    g_banked = per_slot("ll_banked", low_latency=True, count=1, bank_capacity=(N_CLS, 0))[0]

    def bound_fixed(i):
        lr, ious, feat = single[i % K]
        return g_bound.replay(lr_masks=lr, pred_ious=ious, tar_feat=feat)

    ll_modes = {"banked_graph_switching_banks": lambda i: banked(g_banked, i), "bound_graph_one_bank": bound_fixed}
    ll_bad = [i for i in range(B) if not same(banked(g_banked, i).get(), eager(i, "ll", low_latency=True).get())]
    stage._use_bank(banks[0])  # (the bound graph's bank: no re-capture in the timed loop)
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

    rec = dict(tool="tools/bank_switch_throughput.py", card=card(), resident_sets=K, streams=S, banks=B,
               bank_shape=dict(classes=N_CLS, shots=SHOTS), rounds=args.rounds, recapture_rounds=args.recapture_rounds,
               reps=args.reps, masks=N_MASKS, feat_dim=FEAT, num_out_instance=num_out, out_hw=HW,
               outputs_equal_eager=dict(images=K, mismatches=bad, banked_1203_identical=identical_1203,
                                        low_latency_mismatches=ll_bad),
               throughput=res, low_latency_one_image=res_ll,
               timing="CUDA events on the launching stream; inputs resident in HBM, rotating over the sets; the bank "
                      "changes every image; graphs per stream slot; modes alternate in one session")
    print(json.dumps(rec))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")
    if bad or ll_bad:
        raise SystemExit(f"outputs differ from the eager stage: {bad}, low latency {ll_bad}")


if __name__ == "__main__":
    main()
