#!/usr/bin/env python
"""Benchmark of the B200 reference-matching stage (BASELINE.json metric: matching-stage images/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One process per GPU (the driver launches torchrun for N>1; RANK/LOCAL_RANK/WORLD_SIZE from the env).  Every run
executes the reference's three stages through the repository's own host code:

  1. fill      the memory bank (80 classes x L shots, DINOv2 ViT-L features 37x37x1024) is filled from synthetic
               reference shots sharded over the ranks like the reference's DistributedSampler does
               (`MemoryBank.fill_batch`), resolved with ONE NCCL all-reduce (`MemoryBank.sync_fill`) and post-processed.
               L = 10 at N=1 (BASELINE configs[1]) and 30 at N>1 (configs[2], "NCCL memory-bank fill").  -> `fill` record
  2. scoring   256 synthetic images (1024 candidate masks of 256x256 logits, 1024x1024 output, top-100 instances) are
               assigned to ranks by `sharding.shard_indices`; prototypes come from the bank filled in (1).
               A "step" = `--images-per-step` images per GPU (the rank cycles through its shard), `--streams` images in
               flight, every image one CUDA-graph replay of the whole stage; no data-path collective (weak scaling).
  3. collect   one pass of every rank over its shard through `Sam2MatchingBaselineNoAMG.forward` driven by
               `MatcherRunner` (the reference's bs=1, synchronise-per-image test_step), results as COCO RLE, gathered
               on rank 0 with `sharding.collect_results`.                                    -> `forward_api` record

Printed JSON (rank 0, one line):
  value      images/s, inputs already resident in HBM, max-over-ranks device time (CUDA events)
  e2e        images/s through the public API with PINNED HOST inputs and outputs: every step copies its
             logits / IoUs / features host->device and the result device->host inside the timed region
  roofline   dominant kernel (lowres_pack: the single pass over the 268 MB of logits) vs measured HBM peak
  cpu_baseline  the oracle's torch port of the reference stage on the host cores (bounded sample)
`--impl reference` times that same port as the reference arm (rank 0 only).
"""
from __future__ import annotations

import argparse
import contextlib
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "matching_stage_images_per_s"
UNIT = "images/s"
N_IMAGES = 256  # BASELINE configs[2]: "256 synthetic images sharded at 1/2/4/8"
WORKLOAD = dict(workload="coco80x10_sam2L_dinov2L_1024masks_1024x1024", n_masks=1024, lowres=256, feat_hw=37,
                feat_dim=1024, n_classes=80, shots=10, ori_hw=[1024, 1024], num_out_instance=100, nms_thr=0.5,
                n_images=N_IMAGES)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the resident measurement (`value`); the e2e "
                    "legs time min(steps, 10) steps of their own, at least 2, and report that number")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--images-per-step", type=int, default=256, help="images per step per GPU")
    ap.add_argument("--streams", type=int, default=16, help="images in flight per GPU")
    ap.add_argument("--cpu-sample", type=int, default=2, help="images timed for cpu_baseline (0 = skip)")
    ap.add_argument("--n-masks", type=int, default=WORKLOAD["n_masks"])
    ap.add_argument("--n-classes", type=int, default=WORKLOAD["n_classes"], help="other BASELINE configs: 1203 = LVIS-shape "
                    "bank (config 4); --n-masks 4096 = points_per_side 64 (config 5); the default is config 2 / 3")
    ap.add_argument("--n-images", type=int, default=N_IMAGES, help="size of the sharded synthetic dataset")
    ap.add_argument("--no-graph", action="store_true", help="enqueue every kernel from the host instead of replaying "
                    "the captured CUDA graph of the stage")
    ap.add_argument("--tune", action="append", default=[], metavar="NAME=VALUE",
                    help="context tunable for A/B runs (MatchingStage.TUNABLES), e.g. upsample_stage_bytes=0")
    ap.add_argument("--value-only", action="store_true", help="A/B helper: fill + `value` only, short line "
                    "(no e2e legs, no roofline / cpu_baseline) - not the driver's contract line")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned as "
                    "DIR/<name>.npy (rank 0's images; see dump_outputs) to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def configure_workload(args, world):
    shots = 10 if world == 1 else 30
    # every rank keeps its shard resident: bound it to 42 % of the GPU's memory (config 2: 256 x 268 MB = 38 %), the rest
    # is workspaces, outputs and the e2e legs.  A workload with bigger images (config 5: 1.07 GB each) gets a smaller
    # dataset instead of an out-of-memory box; the line says so.
    per_image = 4 * args.n_masks * 65536 + 4 * 1369 * 1024
    total = torch.cuda.get_device_properties(0).total_memory if torch.cuda.is_available() else 192 << 30
    fit = max(16, int(0.42 * total / per_image) // 16 * 16)
    if -(-args.n_images // world) > fit:
        WORKLOAD["n_images_requested"] = args.n_images
        args.n_images = fit * world
    WORKLOAD.update(n_classes=args.n_classes, n_masks=args.n_masks, shots=shots, n_images=args.n_images)
    WORKLOAD["workload"] = (f"coco{args.n_classes}x{shots}_sam2L_dinov2L_{args.n_masks}masks_1024x1024_"
                            f"{args.n_images}img_sharded")
    return dict(WORKLOAD, images_per_step_per_gpu=args.images_per_step,
                l2_policy=f"inputs larger than L2: every rank cycles through its shard of {args.n_images} distinct "
                          f"images x {4 * args.n_masks * 65536 / 1e6:.0f} MB of logits")


def bind_to_gpu_cpus(index: int):
    """Pin this process to the CPUs NVML reports as local to GPU `index`, so that the pinned staging buffers of the e2e
    legs are allocated on the GPU's own NUMA node (one process per GPU: with eight ranks pulling their inputs through one
    socket's memory controllers the box delivers 115 GB/s of H2D in total).  Returns what was done, for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
        handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
        words = pynvml.nvmlDeviceGetCpuAffinity(handle, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return "no local cpus reported"
        os.sched_setaffinity(0, cpus)
        return f"{len(cpus)} cpus local to gpu {phys}"
    except Exception as exc:  # NVML or the affinity call unavailable: run unpinned
        return f"unavailable ({type(exc).__name__})"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1] or [r for _, r in self.rows[-3:]]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            parts = [p.strip() for p in r.split(",")]
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except Exception:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def cpu_port_seconds(images, feats_ins_avg, n_images, timings=None):
    """The oracle's torch port of the reference stage on the host cores; returns seconds per image."""
    from oracle import ref_torch
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = ref_torch.StageConfig(num_out_instance=WORKLOAD["num_out_instance"], nms_thr=WORKLOAD["nms_thr"])
    ts = []
    with torch.inference_mode():
        for i in range(n_images):
            lr, iou, feat = images[i % len(images)]
            t0 = time.perf_counter()
            ref_torch.match_image(lr, iou, feat, feats_ins_avg, cfg, tuple(WORKLOAD["ori_hw"]), timings=timings)
            ts.append(time.perf_counter() - t0)
    return ts


def stage_floor(n_masks, us_per_image):
    """SURVEY.md §8d compulsory-traffic floor of the whole stage (factored pooling => HBM term only)."""
    n, p, e, c, n_cls = n_masks, WORKLOAD["lowres"] ** 2, WORKLOAD["feat_hw"] ** 2, WORKLOAD["feat_dim"], WORKLOAD["n_classes"]
    k, k_out = min(8 * WORKLOAD["num_out_instance"], n), WORKLOAD["num_out_instance"]
    hw = WORKLOAD["ori_hw"][0] * WORKLOAD["ori_hw"][1]
    nbytes = 4 * n * p + 4 * e * c + 4 * n_cls * c + 4 * k * p + 2 * k * hw // 8 + k_out * hw
    peak, _ = measured_peak()
    floor_us = nbytes / (peak * 1e9) * 1e6
    return dict(compulsory_bytes=nbytes, floor_us=floor_us, achieved_us=us_per_image, frac=floor_us / us_per_image)


DUMP_BYTES = 64 << 20  # what --dump-outputs may write in all: half for the per-image arrays, half for the mask sample
DUMP_PIXELS = 4096     # sampled pixels per output mask (fewer when many stream slots share the half)


def dump_outputs(out_dir, last_step, num_out, seed=0):
    """Write what the last timed step returned to its caller as float `.npy` files, so that two builds can be
    compared output for output on the same seeded inputs.

    `last_step`: (image, stream slot, PendingResult) in launch order.  For every distinct image (its last result; a
    seeded sample of the images if there are too many): `scores`, `labels`, `bboxes`, `index` [images, num_out(, 4)],
    NaN past the image's n_out, `counts` [images, 3] = (n_keep, n_sel, n_out) and `image`, the image's index in the
    synthetic dataset.  Masks share one buffer per stream slot, so only the last image of each slot still holds its
    masks: for those images (`mask_image`), `mask_area` [.., num_out] and `mask_samples` [.., num_out, P], the masks
    at the P flat pixel indices `mask_pixels` drawn with a fixed seed, NaN past n_out."""
    import numpy as np
    last = {img: r for r, (img, _, _) in enumerate(last_step)}
    rows = sorted(last.values())
    row_bytes = num_out * (4 + 8 + 32 + 8) + 32
    if len(rows) * row_bytes > DUMP_BYTES // 2:
        pick = np.random.default_rng(seed + 1).choice(len(rows), DUMP_BYTES // 2 // row_bytes, replace=False)
        rows = [rows[i] for i in sorted(pick)]
    mask_rows = sorted({slot: r for r, (_, slot, _) in enumerate(last_step)}.values())
    res = {r: last_step[r][2].get() for r in set(rows) | set(mask_rows)}
    ori_hw = last_step[0][2].ori_hw

    def padded(values, shape, dtype):
        out = np.full(shape, np.nan, dtype)
        for i, v in enumerate(values):
            out[i, :len(v)] = v
        return out

    n = len(rows)
    arrays = dict(
        image=np.array([last_step[r][0] for r in rows], np.float64),
        counts=np.array([[res[r]["counts"][k] for k in ("n_keep", "n_sel", "n_out")] for r in rows], np.float64),
        scores=padded([res[r]["scores"].cpu().numpy() for r in rows], (n, num_out), np.float32),
        labels=padded([res[r]["labels"].cpu().numpy() for r in rows], (n, num_out), np.float64),
        bboxes=padded([res[r]["bboxes"].cpu().numpy() for r in rows], (n, num_out, 4), np.float64),
        index=padded([res[r]["index"].cpu().numpy() for r in rows], (n, num_out), np.float64))
    hw, m_img = ori_hw[0] * ori_hw[1], len(mask_rows)
    n_pix = min(DUMP_PIXELS, hw, (DUMP_BYTES // 2 - 8 * m_img * (num_out + 1)) // (4 * m_img * num_out + 8))
    pixels = np.sort(np.random.default_rng(seed).choice(hw, n_pix, replace=False))
    idx = torch.from_numpy(pixels).to(res[mask_rows[0]]["bboxes"].device)
    areas, samples = [], []
    for r in mask_rows:
        m = res[r]["binary_masks"]
        m = m.reshape(m.shape[0], hw)
        areas.append(m.sum(1).cpu().numpy())
        samples.append(m[:, idx].cpu().numpy())
    arrays.update(mask_image=np.array([last_step[r][0] for r in mask_rows], np.float64),
                  mask_area=padded(areas, (len(mask_rows), num_out), np.float64),
                  mask_samples=padded(samples, (len(mask_rows), num_out, n_pix), np.float32),
                  mask_pixels=pixels.astype(np.float64))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return arrays


def cpu_synthetic(args):
    """CPU-generated images + bank for the CPU legs (the CPU generator of `synth`, as in the parity tests)."""
    synth = importlib.import_module("no-time-to-train_b200.synth")
    inp = synth.make_stage_inputs(args.n_masks, WORKLOAD["feat_dim"], WORKLOAD["n_classes"], WORKLOAD["shots"],
                                  tuple(WORKLOAD["ori_hw"]), seed=1234, clustered=True)
    return [(inp.lr_masks, inp.pred_ious, inp.tar_feat)], inp.feats_ins_avg


def run_reference(args, rank, config):
    """Reference arm: the reference's CPU implementation of the path (oracle port; the reference is Python and
    cannot travel to the GPU box), all host threads, each step a bounded sample of ONE image of the workload."""
    if rank != 0:
        return
    images, bank = cpu_synthetic(args)
    cpu_port_seconds(images, bank, 1)  # one warm-up image is enough on the CPU
    ts = cpu_port_seconds(images, bank, args.steps)
    total = sum(ts)
    value = args.steps / total
    cores = os.cpu_count() or 1
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * total / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f32", data="synthetic", impl="reference", config=config,
                cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind="port",
                                  sample=f"{args.steps} steps of ONE image each (bounded sample of the "
                                         f"{config['images_per_step_per_gpu']}-image step), torch CPU ops, {cores} threads"),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------
# stage 1: memory-bank fill (BASELINE configs[2]: sharded fill + ONE NCCL all-reduce)
# ----------------------------------------------------------------------------------------------------------
def run_fill(pkg, dev, rank, world, dist, centres, fill_batch=16):
    """Returns (bank, record).  Reference shots are strided over the ranks like the DistributedSampler does
    (`COCOMemoryFillDataset` yields L consecutive items per class, `coco_ref_dataset.py:348-361`)."""
    synth = pkg.synth
    n_cls, shots, c = WORKLOAD["n_classes"], WORKLOAD["shots"], WORKLOAD["feat_dim"]
    eh = ew = WORKLOAD["feat_hw"]
    order = [(ci, li) for ci in range(n_cls) for li in range(shots)]
    mine = order[rank::world]

    def batches(items):
        for i in range(0, len(items), fill_batch):
            part = items[i:i + fill_batch]
            pairs = [synth.make_ref_shot_device(ci, li, centres, dev) for ci, li in part]
            yield [ci for ci, _ in part], torch.stack([f for f, _ in pairs]), torch.stack([m for _, m in pairs])

    resident = list(batches(mine))  # this rank's shots, resident in HBM before the timed region
    lib = pkg._lib.load()

    def new_bank(local_only=False):
        b = pkg.MemoryBank(dict(category_num=n_cls, length=shots, feat_shape=(eh * ew, c))).to(dev)
        if local_only:
            b.distributed = False
        return b

    # warm-up on a throw-away bank (kernel load, NCCL channel setup for this message size)
    warm = new_bank()
    for cats, f, m in resident[:2]:
        warm.fill_batch(cats, f, m, (eh, ew))
    warm.sync_fill()
    warm.postprocess()
    del warm
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize(dev)

    bank = new_bank()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    c0 = lib.nttt_launch_count()
    ev[0].record()
    for cats, f, m in resident:
        bank.fill_batch(cats, f, m, (eh, ew))
    ev[1].record()
    bank.sync_fill()           # class-log all_gather, one scatter kernel, ONE all-reduce of [feats_sum | mask_sum]
    ev[2].record()
    bank.postprocess()
    ev[3].record()
    torch.cuda.synchronize(dev)
    launches = int(lib.nttt_launch_count() - c0)
    pool_ms, sync_ms, post_ms = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3])
    ar_us = ar_masks_us = None
    info = bank.last_sync
    if info.get("events"):
        t0, t1, t2 = info["events"]
        ar_us, ar_masks_us = 1e3 * t0.elapsed_time(t1), 1e3 * t1.elapsed_time(t2)
    times = torch.tensor([pool_ms, sync_ms, post_ms, pool_ms + sync_ms + post_ms, ar_us or 0.0], device=dev)
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    pool_ms, sync_ms, post_ms, fill_ms, ar_us_max = times.tolist()

    # the model's bs=1 path (one `fill` call per shot, as `forward_fill_memory` issues them), local bank, bounded sample
    solo = new_bank(local_only=True)
    sample = [(ci, f[j], m[j]) for cats, f, m in resident[:4] for j, ci in enumerate(cats)]  # <= 64 shots of `mine`
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for ci, f, m in sample:
        solo.fill(ci, f, m, (eh, ew))
    e1.record()
    torch.cuda.synchronize(dev)
    bs1_us = 1e3 * e0.elapsed_time(e1) / max(len(sample), 1)
    del solo

    # bit-identity: every rank refills a LOCAL bank with ALL shots in the reference's arrival order (step-major,
    # rank-minor == dataset order) and compares every buffer the test path reads
    local = new_bank(local_only=True)
    for cats, f, m in batches(order):
        local.fill_batch(cats, f, m, (eh, ew))
    local.postprocess()
    same = all(torch.equal(getattr(bank, k), getattr(local, k))
               for k in ("feats_sum", "mask_sum", "masks", "fill_counts", "feats_ins_avg", "feats_avg"))
    flag = torch.tensor([1 if same else 0], device=dev)
    if dist is not None:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    del local, resident
    n_shots = len(order)
    record = dict(shots=n_shots, shots_per_rank=len(mine), n_classes=n_cls, shots_per_class=shots, feat_dim=c,
                  shots_per_launch=fill_batch, fill_ms=fill_ms, pool_ms=pool_ms, sync_ms=sync_ms, postprocess_ms=post_ms,
                  per_shot_us=1e3 * fill_ms / n_shots, per_local_shot_us=1e3 * pool_ms / max(len(mine), 1),
                  bs1_per_shot_us=bs1_us,
                  allreduce_us=ar_us_max if world > 1 else None, allreduce_bytes=info.get("allreduce_bytes") if world > 1 else 0,
                  masks_allreduce_us=ar_masks_us, masks_allreduce_bytes=info.get("masks_allreduce_bytes") if world > 1 else 0,
                  class_log_bytes=info.get("class_log_bytes") if world > 1 else 0,
                  collectives="1 all_gather (class log) + 1 all_reduce (feats_sum|mask_sum) + 1 all_reduce (low-res masks, "
                              "state-dict only)" if world > 1 else "none (single process)",
                  bit_identical_across_world=bool(flag.item()), kernel_launches=launches,
                  timing="CUDA events on the launching stream, max over ranks; inputs resident in HBM")
    return bank, record


# ----------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    config = configure_workload(args, world)
    if args.impl == "reference":
        run_reference(args, rank, config)
        return

    pkg = importlib.import_module("no-time-to-train_b200")
    ops = importlib.import_module("no-time-to-train_b200.ops")
    sharding = importlib.import_module("no-time-to-train_b200.sharding")
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU path)"
    nttt_env = {k: v for k, v in os.environ.items() if k.startswith("NTTT_")}
    lib = pkg._lib.load()
    if lib.nttt_build_is_ablation() and not args.value_only:
        raise SystemExit("libnttt_b200.so is an ablation build (NTTT_BUILD_ABLATE): rebuild the product library for a "
                         "contract bench line")
    if "NTTT_STOP_AFTER" in nttt_env and not args.value_only:
        raise SystemExit("NTTT_STOP_AFTER is set: refusing to print a contract bench line for a truncated pipeline")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # (N > 1 only: at N = 1 the cpu_baseline leg wants every host core)
    numa = bind_to_gpu_cpus(local_rank) if world > 1 else "not bound (single process)"  # before any pinned allocation
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL may print its version banner on fd 1 at communicator creation; stdout must carry exactly one JSON
        # line, so route fd 1 to stderr until the first collective has run.
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    synth = pkg.synth
    centres = synth.cluster_centres(WORKLOAD["feat_dim"])
    ori_hw = tuple(WORKLOAD["ori_hw"])
    n_out = WORKLOAD["num_out_instance"]

    # ---- stage 1: fill + one all-reduce + post-process --------------------------------------------------
    bank, fill_record = run_fill(pkg, dev, rank, world, dist, centres)

    # ---- stage 2: scoring; this rank's shard of the dataset, resident in HBM ------------------------------
    shard = sharding.shard_indices(args.n_images, rank, world)
    distinct = list(dict.fromkeys(shard))  # the sampler pads by repetition; hold every image once
    resident = {i: synth.make_stage_inputs_device(args.n_masks, centres, dev, seed=1234 + i) for i in distinct}
    B, S = args.images_per_step, max(1, min(args.streams, args.images_per_step, len(shard)))
    stage = pkg.MatchingStage(dev, pkg.StageConfig(nms_thr=WORKLOAD["nms_thr"], num_out_instance=n_out,
                                                   enc_hw=(WORKLOAD["feat_hw"], WORKLOAD["feat_hw"])))
    stage.set_prototypes(bank.feats_ins_avg)
    for item in args.tune:
        name, val = item.split("=")
        stage.tune(name, int(val))
    streams = [torch.cuda.Stream(dev) for _ in range(S)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # one eager image to count the kernels of a stage invocation (graph replays do not pass through the C counter)
    stage.match_async(*resident[shard[0]], ori_hw, slot=0)  # (first call: also builds the antialias tables)
    torch.cuda.synchronize(dev)
    c0 = lib.nttt_launch_count()
    stage.match_async(*resident[shard[0]], ori_hw, slot=0, persistent_out=None)
    torch.cuda.synchronize(dev)
    launches_per_image = int(lib.nttt_launch_count() - c0)

    use_graph = not args.no_graph
    # Persistent output buffers, one per stream slot: consecutive images of a slot are DIFFERENT images, so the sparse
    # unpack always clears one image's rectangles and writes another's (never the same rect twice in a row).
    outs = [(torch.zeros((n_out, *ori_hw), dtype=torch.uint8, device=dev),
             torch.zeros((n_out, 4), dtype=torch.int32, device=dev)) for _ in range(S)]
    graphs = {}
    if use_graph:
        # the public API's graph mode; one graph per resident image (its tensors ARE the static inputs), sharing the
        # workspace and the output buffers of its stream slot
        for pos, i in enumerate(shard):
            if (i, pos % S) in graphs:
                continue
            g = stage.graphed(args.n_masks, WORKLOAD["feat_dim"], ori_hw, key=("bench", pos % S),
                              persistent_out=outs[pos % S])
            g.lr_masks, g.pred_ious, g.tar_feat = resident[i]
            graphs[(i, pos % S)] = g.capture()

    last_step = []  # (image, slot, result) of every image of the most recent step, for --dump-outputs

    def resident_step():
        last_step.clear()
        for b in range(B):
            pos = b % len(shard)
            k = pos % S
            with torch.cuda.stream(streams[k]):
                if use_graph:
                    pend = graphs[(shard[pos], k)].replay()
                else:
                    pend = stage.match_async(*resident[shard[pos]], ori_hw, slot=k, persistent_out=outs[k])
            last_step.append((shard[pos], k, pend))

    def timed(step_fn, steps):
        barrier()
        cur = torch.cuda.current_stream(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(cur)
        for s in streams:
            s.wait_event(e0)
        for _ in range(steps):
            step_fn()
        for s in streams:
            cur.wait_stream(s)
        e1.record(cur)
        barrier()
        t1 = time.perf_counter()
        mine = torch.tensor([e0.elapsed_time(e1)], device=dev)
        per_rank = [mine.clone() for _ in range(world)]
        if dist is not None:
            dist.all_gather(per_rank, mine)
        per_rank = [float(t.item()) for t in per_rank]
        return max(per_rank), t0, t1, per_rank

    warmup = max(args.warmup, 3)
    for _ in range(warmup):
        resident_step()
    torch.cuda.synchronize(dev)
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ms_total, t0, t1, ms_per_rank = timed(resident_step, args.steps)
    clock_info = clocks.stop(t0, t1) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_step, n_out)
    launches = launches_per_image * args.steps * B
    images = world * args.steps * B
    value = images / (ms_total / 1e3)
    us_per_image = 1e3 * ms_total / (args.steps * B)

    if args.value_only:
        if rank == 0:
            print(json.dumps(dict(metric=METRIC, value_only=True, value=value, us_per_image=us_per_image, n_gpus=world,
                                  steps=args.steps, images_per_step_per_gpu=B, streams=S, clocks=clock_info,
                                  ms_per_rank=ms_per_rank, fill=fill_record, env=nttt_env, tune=args.tune)))
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- e2e: pinned host inputs -> device -> stage -> pinned host outputs, every step ----------------------
    E2E_B = 16
    host = [tuple(t.cpu().pin_memory() for t in resident[shard[p % len(shard)]]) for p in range(min(E2E_B, len(distinct)))]
    Se = min(S, E2E_B)
    out_host = [dict(masks=torch.empty((n_out, *ori_hw), dtype=torch.bool).pin_memory(),
                     boxes=torch.empty((n_out, 4), dtype=torch.int64).pin_memory(),
                     scores=torch.empty((n_out,), dtype=torch.float32).pin_memory(),
                     labels=torch.empty((n_out,), dtype=torch.int64).pin_memory(),
                     counts=torch.empty((4,), dtype=torch.int32).pin_memory()) for _ in range(Se)]
    dev_in = [tuple(torch.empty_like(t, device=dev) for t in host[0]) for _ in range(Se)]
    h2d = sum(t.numel() * t.element_size() for t in host[0]) * E2E_B
    d2h = sum(t.numel() * t.element_size() for t in out_host[0].values()) * E2E_B

    e2e_graphs = []
    if use_graph:
        for k in range(Se):
            g = stage.graphed(args.n_masks, WORKLOAD["feat_dim"], ori_hw, key=("e2e", k))
            g.lr_masks, g.pred_ious, g.tar_feat = dev_in[k]
            e2e_graphs.append(g.capture())

    def e2e_step():
        for i in range(E2E_B):
            k = i % Se
            with torch.cuda.stream(streams[k]):
                for dst, src in zip(dev_in[k], host[i % len(host)]):
                    dst.copy_(src, non_blocking=True)
                p = e2e_graphs[k].replay() if use_graph else stage.match_async(*dev_in[k], ori_hw, slot=("e2e", k))
                oh = out_host[k]
                oh["masks"].copy_(p.masks, non_blocking=True)
                oh["boxes"].copy_(p.boxes, non_blocking=True)
                oh["scores"].copy_(p.scores, non_blocking=True)
                oh["labels"].copy_(p.labels, non_blocking=True)
                oh["counts"].copy_(p.counts, non_blocking=True)

    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize(dev)
    e2e_steps = max(2, min(args.steps, 10))
    ms_e2e, _, _, _ = timed(e2e_step, e2e_steps)
    e2e_value = world * e2e_steps * E2E_B / (ms_e2e / 1e3)

    # ---- e2e_rle: same, but the result leaves the device as COCO RLE strings (fused nttt_rle_encode) instead of the
    # dense bool masks: what the reference's _output_inqueue/encode_results ultimately produce (SURVEY.md §8f rank 1)
    e2e_rle = None
    if use_graph:
        cap_chars = stage.cfg.rle_cap_chars
        rle_host = [dict(chars=torch.empty((n_out, cap_chars), dtype=torch.uint8).pin_memory(),
                         n_chars=torch.empty((n_out,), dtype=torch.int32).pin_memory(),
                         boxes=torch.empty((n_out, 4), dtype=torch.int64).pin_memory(),
                         scores=torch.empty((n_out,), dtype=torch.float32).pin_memory(),
                         labels=torch.empty((n_out,), dtype=torch.int64).pin_memory(),
                         counts=torch.empty((4,), dtype=torch.int32).pin_memory()) for _ in range(Se)]
        rle_graphs = []
        for k in range(Se):
            g = stage.graphed(args.n_masks, WORKLOAD["feat_dim"], ori_hw, key=("e2e_rle", k), rle=True, dense_masks=False)
            g.lr_masks, g.pred_ious, g.tar_feat = dev_in[k]
            rle_graphs.append(g.capture())
        d2h_rle = sum(t.numel() * t.element_size() for t in rle_host[0].values()) * E2E_B

        def e2e_rle_step():
            for i in range(E2E_B):
                k = i % Se
                with torch.cuda.stream(streams[k]):
                    for dst, src in zip(dev_in[k], host[i % len(host)]):
                        dst.copy_(src, non_blocking=True)
                    p = rle_graphs[k].replay()
                    oh = rle_host[k]
                    oh["chars"].copy_(p.rle[2], non_blocking=True)
                    oh["n_chars"].copy_(p.rle[3], non_blocking=True)
                    oh["boxes"].copy_(p.boxes, non_blocking=True)
                    oh["scores"].copy_(p.scores, non_blocking=True)
                    oh["labels"].copy_(p.labels, non_blocking=True)
                    oh["counts"].copy_(p.counts, non_blocking=True)

        for _ in range(2):
            e2e_rle_step()
        torch.cuda.synchronize(dev)
        ms_rle, _, _, _ = timed(e2e_rle_step, e2e_steps)
        n_live = int(rle_host[0]["counts"][2])
        lens = rle_host[0]["n_chars"][:n_live]
        e2e_rle = dict(value=world * e2e_steps * E2E_B / (ms_rle / 1e3), unit=UNIT, h2d_bytes_per_step=h2d,
                       d2h_bytes_per_step=d2h_rle, steps=e2e_steps, images_per_step_per_gpu=E2E_B,
                       rle_bytes_per_image=int(lens.sum()), rle_overflow=bool((lens < 0).any() or (lens > cap_chars).any()))
        del rle_graphs
    del e2e_graphs

    # ---- stage 3: the drop-in class driven like the reference drives it (bs=1, sync per image), results gathered ----
    class SeamModel(pkg.Sam2MatchingBaselineNoAMG):
        """Encoder seams answered from the resident synthetic tensors (the frozen encoders are out of scope)."""

        def _extract_target_features(self, tar_img, device):
            return resident[self._cur][2], tar_img

        def _forward_sam(self, imgs):
            lr, iou, _ = resident[self._cur]
            return lr, iou, None

    class Dataset:
        def __len__(self):
            return args.n_images

        def __getitem__(self, i):
            model._cur = i
            return dict(target_img=torch.zeros(3, 8, 8), target_img_info=dict(ori_height=ori_hw[0], ori_width=ori_hw[1],
                                                                              file_name=f"synthetic_{i}", id=i))

    model = SeamModel(sam2_infer_cfgs=dict(points_per_side=32, testing_point_bs=256, iou_thr=0.0, nms_thr=WORKLOAD["nms_thr"],
                                           num_out_instance=n_out, kmeans_k=2, n_pca_components=2, cls_num_per_mask=1),
                      memory_bank_cfg=dict(enable=True, category_num=WORKLOAD["n_classes"], length=WORKLOAD["shots"]),
                      encoder_geometry=(518, 14, WORKLOAD["feat_dim"]), device=dev)
    model.memory_bank.load_state_dict(bank.state_dict())
    runner = pkg.MatcherRunner(model, "test", Dataset(), rle=True)
    barrier()
    tw0 = time.perf_counter()
    runner.run()
    torch.cuda.synchronize(dev)
    tw1 = time.perf_counter()
    with contextlib.redirect_stdout(sys.stderr):
        gathered = runner.after_test()
    tw2 = time.perf_counter()
    lat = torch.tensor([sum(runner.time_queue) / max(len(runner.time_queue), 1), tw1 - tw0], device=dev)
    if dist is not None:
        dist.all_reduce(lat, op=dist.ReduceOp.MAX)
    forward_api = None
    if rank == 0:
        ids = [r[0]["image_id"] if r else None for r in gathered["results"]]
        forward_api = dict(images=len(gathered["results"]), instances=len(gathered["results_unpacked"]),
                           images_per_s=args.n_images / float(lat[1]), forward_ms_per_image=1e3 * float(lat[0]),
                           collect_ms=1e3 * (tw2 - tw1),
                           ordered=all(i is None or i == k for k, i in enumerate(ids)) and len(ids) == args.n_images,
                           note="Sam2MatchingBaselineNoAMG.forward through MatcherRunner: bs=1, device synchronise "
                                "around every image as in sam2matcher_pl.py:178-191, results as device-encoded COCO RLE, "
                                "gathered with sharding.collect_results; encoders replaced by resident synthetic tensors")
    del model, runner

    # ---- latency of ONE image (rank 0): the whole stage as one CUDA-graph replay in low-latency mode, the device idle
    #      before every replay, CUDA events around it; the throughput-mode shapes beside it for comparison ---------------
    latency = None
    if rank == 0:
        latency = {}
        for low in (True, False):
            g = stage.graphed(args.n_masks, WORKLOAD["feat_dim"], ori_hw, key=("latency", low), low_latency=low)
            first = resident[distinct[0]]
            g.lr_masks.copy_(first[0]); g.pred_ious.copy_(first[1]); g.tar_feat.copy_(first[2])
            g.capture()
            times = []
            for rep in range(28):
                img = resident[distinct[rep % min(8, len(distinct))]]
                g.lr_masks.copy_(img[0]); g.pred_ious.copy_(img[1]); g.tar_feat.copy_(img[2])
                torch.cuda.synchronize(dev)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); g.replay(); e1.record()
                torch.cuda.synchronize(dev)
                times.append(1e3 * e0.elapsed_time(e1))
            times = sorted(times[4:])
            latency["low_latency_us" if low else "throughput_shapes_us"] = dict(median=times[len(times) // 2], min=times[0])
            del g
        latency["note"] = ("one image alone on an idle device, whole stage = one CUDA-graph replay (nttt_match_args."
                           "low_latency = 1 / 0), CUDA events; inputs in HBM")

    # ---- per-stage share (single stream, CUDA events between the stage's kernels) and the roofline kernel --
    stage_ms = {}
    roofline = None
    if rank == 0:
        stage.profile(True)
        reps = min(16, len(distinct))
        try:
            for rep in range(2 * reps):
                stage.match_async(*resident[distinct[rep % reps]], ori_hw, slot=0, low_latency=True)
                for k, v in stage.profile_read().items():
                    if rep >= reps:
                        stage_ms[k] = stage_ms.get(k, 0.0) + v / reps
        except Exception as exc:
            stage_ms = {"unavailable": 0.0}
            print(f"stage profile unavailable: {exc}", file=sys.stderr)
        stage.profile(False)
        # dominant kernel alone, over inputs larger than L2 (the shard's images rotate), events on the launching stream
        pool = [resident[i][0] for i in distinct[:32]]
        reps = max(3 * len(pool), 48)
        tp_out = ops.threshold_pack(pool[0])
        for t in pool:
            ops.threshold_pack(t, out=tp_out, want_stab=False)
        torch.cuda.synchronize(dev)
        cur = torch.cuda.current_stream(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(cur)
        for i in range(reps):
            ops.threshold_pack(pool[i % len(pool)], out=tp_out, want_stab=False)
        e1.record(cur)
        torch.cuda.synchronize(dev)
        k_ms = e0.elapsed_time(e1) / reps
        alg_bytes = 4 * args.n_masks * WORKLOAD["lowres"] ** 2
        peak, peak_src = measured_peak()
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9
        traffic, traffic_src, prof_kernel = None, None, None
        try:  # DRAM bytes per launch from the committed `ncu --set full` capture of this kernel at this shape
            with open(os.path.join(ROOT, "profiles", "lowres_pack_ncu.json")) as f:
                prof = json.load(f)
            prof_kernel = prof.get("kernel")
            if args.n_masks == 1024:
                traffic, traffic_src = prof["traffic_bytes_per_launch"], "profiles/lowres_pack_ncu.json (ncu --set full capture)"
        except Exception:
            pass
        persistent = not any(t.split("=") == ["lowres_persistent", "0"] for t in args.tune)
        roofline = dict(bound="hbm", kernel=prof_kernel if persistent and prof_kernel else
                        ("lowres_pack_persistent_kernel<3>" if persistent else "lowres_pack_fast_kernel"), achieved=achieved, peak=peak, unit="GB/s",
                        frac=achieved / peak, traffic=traffic, traffic_source=traffic_src, peak_source=peak_src,
                        alg_bytes_per_launch=alg_bytes, us_per_launch=1e3 * k_ms,
                        note="launches back to back on one stream over rotating images; peak is the driver's COPY "
                             "bandwidth (read+write) - a read-only stream can exceed it (frac > 1 at 4096 masks, where "
                             "the persistent kernel's 296 CTAs run 14 masks each)")

    # ---- CPU baseline (rank 0, N=1 only): the oracle's torch port on a bounded sample -------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and args.cpu_sample > 0:
        images_cpu = [tuple(t.cpu() for t in resident[shard[0]])]
        bank_cpu = bank.feats_ins_avg.cpu()
        cpu_port_seconds(images_cpu, bank_cpu, 1)
        tm = {}
        ts = cpu_port_seconds(images_cpu, bank_cpu, args.cpu_sample, timings=tm)
        cores = os.cpu_count() or 1
        cpu_baseline = dict(value=len(ts) / sum(ts), unit=UNIT, cores=cores, kind="port",
                            sample=f"{len(ts)} image(s) of the same workload after 1 warm-up, torch CPU ops, "
                                   f"{cores} threads",
                            ms_per_stage={k: 1e3 * v / len(ts) for k, v in tm.items()})

    if rank == 0:
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=warmup,
                    ms_per_step=ms_total / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f32", data="synthetic", config=config,
                    run=dict(streams=S, launch="cuda_graph_replay" if use_graph else "host_enqueue",
                             images_resident_per_gpu=len(distinct), timed_region_ms=ms_total, ms_per_rank=ms_per_rank,
                             env=nttt_env, tune=args.tune, cpu_affinity=numa),
                    us_per_image=us_per_image,
                    e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                             steps=e2e_steps, images_per_step_per_gpu=E2E_B),
                    e2e_rle=e2e_rle, fill=fill_record, forward_api=forward_api, gpu_launches=int(launches),
                    clocks=clock_info, roofline=roofline, cpu_baseline=cpu_baseline, latency=latency,
                    stage_us_per_image={k: 1e3 * v for k, v in stage_ms.items()},
                    stage_us_note="one image at a time on one stream, low-latency launch shapes, host-enqueued (launch "
                                  "gaps included); with images in flight the stages cost what DESIGN.md §5 lists as marginals",
                    stage_roofline=stage_floor(args.n_masks, us_per_image))
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
