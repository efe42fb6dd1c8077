"""Throughput of the matching stage fed by a producer that allocates fresh input tensors for every image.

    python tools/bound_graph_throughput.py [--sets 32] [--streams 16] [--rounds 40] [--reps 3] [--out FILE.json]

Config-2 shapes (1024 masks, ViT-L features, 80 classes, 1024 x 1024 output), inputs generated on the device.  `--sets`
resident input sets (each a separate allocation, 268 MB of single-plane logits or 1.07 GB of raw decoder output, far
more than the 126 MB of L2 in total) are consumed in rotation, image i on stream slot i % streams.  Graphs are held per
stream slot, not per image.  For single-plane inputs (lr_masks [n,256,256] + pred_ious) and for the decoder's raw output
as 4 per-batch chunks of [256, 4, 256, 256] (+ multi_ious), in images/s (CUDA events on the launching stream around
`--rounds` passes over all sets, after two warm-up passes; the modes alternate in one session, `--reps` times each):

  eager            `match_async` in throughput mode;
  static_copy      a static graph per slot, the inputs `copy_`-ed into its buffers before each replay;
  bound            a bound graph per slot (`graphed(..., bind=True)`), each replay binding the set's own tensors;
  graph_per_set    one static graph per resident set whose buffers ARE that set (bench.py's setup, the reference figure
                   a producer-fed pipeline could not reach before bound graphs).

Also one image at a time in low-latency mode (replay or call, then synchronise), single-plane, in microseconds: the
bound graph on rotating sets, the static graph on its own buffers, and eager calls on rotating sets.

Before timing, every set's outputs of every mode are compared with the eager result: counts, scores (NaN pattern
included), labels, boxes, index and masks must be identical.  The card's name and power limit are read in the same run.
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

N_MASKS, FEAT, N_CLS, M, CHUNK = 1024, 1024, 80, 4, 256
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
    ap.add_argument("--rounds", type=int, default=40, help="timed passes over all sets per measurement")
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
    S, K = args.streams, args.sets
    streams = [torch.cuda.Stream(dev) for _ in range(S)]
    num_out = stage.cfg.num_out_instance

    # ---- resident sets: single-plane (lr_masks, pred_ious, tar_feat); multimask (chunks, multi_ious, tar_feat)
    single = [synth.make_stage_inputs_device(N_MASKS, centres, dev, seed=1234 + i) for i in range(K)]
    multi = []
    for i, (lr, _, feat) in enumerate(single):
        g = torch.Generator(device=dev).manual_seed(5678 + i)
        chunks = []
        for k in range(N_MASKS // CHUNK):  # the decoder's per-batch outputs: separate allocations
            base = lr[k * CHUNK:(k + 1) * CHUNK]
            ch = torch.empty((CHUNK, M, 256, 256), dtype=torch.float32, device=dev)
            for j in range(M):
                shift = 0.35 * (j + 1) * torch.randn((CHUNK, 1, 1), generator=g, device=dev)
                ch[:, j] = base * (1.0 + 0.1 * j) + shift + 0.3 * torch.randn((CHUNK, 256, 256), generator=g, device=dev)
            chunks.append(ch)
        ious = 0.2 + 0.8 * torch.rand((N_MASKS, M), generator=g, device=dev)
        multi.append((chunks, ious, feat))
    torch.cuda.synchronize()

    def outs():
        return [(torch.zeros((num_out, *HW), dtype=torch.uint8, device=dev),
                 torch.zeros((num_out, 4), dtype=torch.int32, device=dev)) for _ in range(S)]

    def kind_kw(kind):
        return dict(n_multi=M, chunk_prompts=CHUNK) if kind == "multi" else {}

    def per_slot(tag, kind, bind, low_latency=False, count=None):
        o = outs()
        return [stage.graphed(N_MASKS, FEAT, HW, key=(tag, s), persistent_out=o[s], low_latency=low_latency, bind=bind,
                              **kind_kw(kind)).capture() for s in range(count or S)]

    def per_set(tag, kind):
        o = outs()
        gs = []
        for i in range(K):
            g = stage.graphed(N_MASKS, FEAT, HW, key=(tag, i % S), persistent_out=o[i % S], **kind_kw(kind))
            if kind == "multi":
                g.lr_masks, g.multi_ious, g.tar_feat = multi[i]
            else:
                g.lr_masks, g.pred_ious, g.tar_feat = single[i]
            gs.append(g.capture())
        return gs

    def eager_call(kind, i, slot, low_latency=False):
        if kind == "multi":
            chunks, ious, feat = multi[i]
            return stage.match_async(chunks, None, feat, HW, slot=slot, multi_ious=ious, low_latency=low_latency)
        return stage.match_async(*single[i], HW, slot=slot, low_latency=low_latency)

    def copy_replay(kind, g, i):
        if kind == "multi":
            chunks, ious, feat = multi[i]
            for dst, src in zip(g.lr_masks, chunks):
                dst.copy_(src)
            g.multi_ious.copy_(ious)
        else:
            lr, ious, feat = single[i]
            g.lr_masks.copy_(lr)
            g.pred_ious.copy_(ious)
        g.tar_feat.copy_(feat)
        return g.replay()

    def bound_replay(kind, g, i):
        if kind == "multi":
            chunks, ious, feat = multi[i]
            return g.replay(lr_masks=chunks, multi_ious=ious, tar_feat=feat)
        lr, ious, feat = single[i]
        return g.replay(lr_masks=lr, pred_ious=ious, tar_feat=feat)

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
        return args.rounds * K / (e0.elapsed_time(e1) / 1e3)

    def on_streams(fn):
        def step():
            for i in range(K):
                with torch.cuda.stream(streams[i % S]):
                    fn(i)
        return step

    res, mism = {}, {}
    for kind in ("single", "multi"):
        static = per_slot(f"static_{kind}", kind, bind=False)
        bound = per_slot(f"bound_{kind}", kind, bind=True)
        pset = per_set(f"perset_{kind}", kind)
        # ---- outputs of every mode == eager, set by set
        bad = []
        for i in range(K):
            ref = eager_call(kind, i, "check").get()
            for name, out in (("static_copy", copy_replay(kind, static[i % S], i).get()),
                              ("bound", bound_replay(kind, bound[i % S], i).get()),
                              ("graph_per_set", pset[i].replay().get())):
                if not same(out, ref):
                    bad.append((i, name))
        mism[kind] = bad
        modes = {"eager": on_streams(lambda i, kind=kind: eager_call(kind, i, ("eager", i % S))),
                 "static_copy": on_streams(lambda i, kind=kind: copy_replay(kind, static[i % S], i)),
                 "bound": on_streams(lambda i, kind=kind: bound_replay(kind, bound[i % S], i)),
                 "graph_per_set": on_streams(lambda i: pset[i].replay())}
        for step in modes.values():
            for _ in range(2):
                step()
        torch.cuda.synchronize()
        got = {k: [] for k in modes}
        for _ in range(args.reps):
            for k, step in modes.items():
                got[k].append(timed(step))
        res[kind] = {k: dict(images_per_s=statistics.median(v), us_per_image=1e6 / statistics.median(v), runs=v)
                     for k, v in got.items()}
        del static, bound, pset
        torch.cuda.synchronize()

    # ---- one image at a time, low-latency launch shapes, single-plane
    g_bound = per_slot("ll_bound", "single", bind=True, low_latency=True, count=1)[0]
    g_static = per_slot("ll_static", "single", bind=False, low_latency=True, count=1)[0]
    g_static.lr_masks.copy_(single[0][0])
    g_static.pred_ious.copy_(single[0][1])
    g_static.tar_feat.copy_(single[0][2])
    ll_modes = {"bound_graph": lambda i: bound_replay("single", g_bound, i % K),
                "static_graph": lambda i: g_static.replay(),
                "eager": lambda i: eager_call("single", i % K, "ll", low_latency=True)}
    ll_bad = [i for i in range(K) if not same(bound_replay("single", g_bound, i).get(),
                                              stage.match(*single[i], HW, low_latency=True))]
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

    rec = dict(tool="tools/bound_graph_throughput.py", card=card(), resident_sets=K, streams=S, rounds=args.rounds,
               reps=args.reps, masks=N_MASKS, feat_dim=FEAT, classes=N_CLS, num_out_instance=num_out, out_hw=HW,
               multimask=dict(planes=M, chunks=N_MASKS // CHUNK, chunk_prompts=CHUNK),
               outputs_equal_eager=dict(sets=K, mismatches=mism, low_latency_mismatches=ll_bad),
               single_plane=res["single"], multimask_chunks=res["multi"], low_latency_one_image=res_ll,
               timing="CUDA events on the launching stream; inputs resident in HBM, rotating over the sets; "
                      "graphs per stream slot except graph_per_set; modes alternate in one session")
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")
    if any(mism.values()) or ll_bad:
        raise SystemExit(f"outputs differ from the eager stage: {mism}, low latency {ll_bad}")


if __name__ == "__main__":
    main()
