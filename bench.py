#!/usr/bin/env python
"""bench.py — image-pairs/sec of the pairwise deep front-end hot path (detect + match + verify).

    python bench.py --gpus N --steps K --warmup W                 # this repo's CUDA path, default workload
    python bench.py --workload {vga_lightglue,mp1_lightglue,seq_superglue,superpoint_only,small_stop}
    python bench.py --impl reference --gpus N --steps K ...        # the reference algorithm on the host CPU cores
    python bench.py --scaling strong --frames F                    # ONE fixed job through the L2 seam, pairs sharded p mod world
    python bench.py --steps K --warmup W --dump-outputs DIR        # also write what the last timed step computed (dump_outputs)

Workloads (config.workload):
  vga_lightglue   (default; the driver's line) steady state of BASELINE.json configs[3] with the deep_front_end.yaml matcher: synthetic
                  640x480 sequence, Sequential(max_frame_lookahead=20), SuperPoint (<= 5000 keypoints) -> LightGlue (9 layers) ->
                  RANSAC-5pt.  One STEP = 2 new frames: 2 detections + 40 matches + 40 verifications.
  mp1_lightglue   configs[2]: 1024x1024 frames, SuperPoint -> LightGlue over all earlier frames.  STEP = 1 detection + 16 pairs.
  seq_superglue   configs[3] verbatim: SuperPoint + SuperGlue (20 Sinkhorn iterations) + RANSAC-5pt.  STEP = 1 new frame + 20 pairs.
  superpoint_only configs[1]: SuperPoint detect + describe only, 640x480.  STEP = 32 frames; metric = images/s.
  small_stop      launch-bound regime: 1024 keypoints, 'stop' weights (early exit at layer 4-5, pruning on).  STEP = 40 pairs.
Pairs shard across GPUs with no data-path collective (one weight broadcast at start-up); per-GPU work is fixed => "weak" scaling.
`--scaling strong` instead times one fixed job (F frames, lookahead 20) through B200CorrespondenceGenerator (two-view verification run under the matching),
including image (re-)detection on every rank and the final gather, wall-clock on rank 0; each of the --steps steps is one whole job.

`value` times the device-resident path (frames already in HBM, features / matches stay in HBM, only per-pair scalars come back);
`e2e` times the same step through the GTSfM plugin classes with HOST numpy buffers, so every H2D / D2H copy the per-call API
implies is inside the timed region (feature cache OFF, the default; `e2e.with_feature_cache` is the opt-in number beside it).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from collections import deque
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

THR_PX = 4.0
FP16_ATTN = False  # set by --fp16-attention
MATCH_BATCH = 8  # pairs per lock-step LightGlue batch (the library maximum)
DETECT_LANES = int(os.environ.get("B2_DETECT_LANES", "4"))  # mirrors gtsfm_b200.pipeline.DETECT_LANES (read there from the same variable)

WORKLOADS = {
    "vga_lightglue": dict(
        H=480, W=640, max_kp=5000, matcher="lightglue", profile="bench", lookahead=20, new_frames=2, verify=True, dominant="k_flash",
        text="SuperPoint+LightGlue+RANSAC-5pt, synthetic 640x480 sequence, Sequential lookahead 20 (BASELINE configs[3] steady state, deep_front_end.yaml matcher)",
        matcher_text="LightGlue 9 layers, full depth (synthetic 'bench' weights: no early exit, nothing pruned)"),
    "mp1_lightglue": dict(
        H=1024, W=1024, max_kp=5000, matcher="lightglue", profile="bench", lookahead=16, new_frames=1, verify=True, dominant="k_flash",
        text="SuperPoint+LightGlue+RANSAC-5pt, synthetic 1024x1024 frames, each new frame against 16 resident frames (BASELINE configs[2]: "
             "the full exhaustive job amortises one detection over 99.5 pairs; 1 per 16 here is pessimistic)",
        matcher_text="LightGlue 9 layers, full depth (synthetic 'bench' weights)"),
    "seq_superglue": dict(
        H=480, W=640, max_kp=5000, matcher="superglue", profile="sharp", lookahead=20, new_frames=1, verify=True, dominant="k_flash",
        text="SuperPoint+SuperGlue+RANSAC-5pt two-view, synthetic 640x480 sequence, Sequential lookahead 20 (BASELINE configs[3] verbatim)",
        matcher_text="SuperGlue 18 layers, 20 Sinkhorn iterations, threshold 0.2 (synthetic 'sharp' weights)"),
    "superpoint_only": dict(
        H=480, W=640, max_kp=5000, matcher=None, profile=None, lookahead=0, new_frames=32, verify=False, dominant="k_conv_ps",
        text="SuperPoint detect+describe only, synthetic 640x480 frames (BASELINE configs[1])", matcher_text="-"),
    "small_stop": dict(
        H=480, W=640, max_kp=1024, matcher="lightglue", profile="stop", lookahead=20, new_frames=2, verify=True, dominant="k_flash",
        text="SuperPoint (1024 keypoints)+LightGlue+RANSAC-5pt, 640x480 sequence, lookahead 20: the launch-/sync-bound regime (early exit + pruning fire)",
        matcher_text="LightGlue 'stop' weights: early exit around layer 4-5, pruning at every layer (reference CPU semantics)"),
}
# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full` captures
# (profiles/): per workload, or None where no capture of that workload's launch shape exists
DOMINANT_DRAM_BYTES = {
    # profiles/r02_flash_ps.txt: the 16-problem launch (self- or cross-attention of a lock-step batch of 8 pairs at 5000 keypoints;
    # 2 of every 3 k_flash_ps launches of this workload have that shape): 2.726 GB read + 0.086 GB written, against 0.33 GB of
    # operands - the 64 heads of a batch do not fit L2 together, K / V tiles are re-read per 256-query block
    "vga_lightglue": 2725897000 + 86424320,
    # profiles/r02_conv_ps_1b.txt: conv1b, the largest of the nine k_conv_ps launch shapes (43 % of the network's FLOPs): input planes once
    "superpoint_only": 78848256 + 5455104,
}


def config_of(name: str) -> dict:
    w = WORKLOADS[name]
    pairs = w["lookahead"] * w["new_frames"]
    return {
        "workload": f"{name}: {w['text']}", "frame": [w["H"], w["W"]], "max_keypoints": w["max_kp"], "lookahead": w["lookahead"],
        "new_frames_per_step": w["new_frames"], "pairs_per_step": pairs, "matcher": w["matcher_text"],
        "match_batch": MATCH_BATCH if w["matcher"] == "lightglue" else 1,
        "attention": "fp16 single-MMA (reference CUDA numerics, opt-in)" if FP16_ATTN else "split-fp16 x3 (fp32-equivalent, parity-pinned default)",
        "ransac": "5pt, 1000 hypotheses, thr 4 px, conf 0.999999" if w["verify"] else "-", "weights": "seeded synthetic (no checkpoint offline)",
        "l2": "256 MiB flush between timed steps", "parallelism": "pairs sharded per GPU, no data-path collective",
        "detect_lanes": (f"{DETECT_LANES} SuperPoint instances on {DETECT_LANES} streams per GPU, frames of a step enqueued without host "
                         "synchronisation (DeviceFrontEnd.detect_many)") if not w["matcher"] else "1 (detect per new frame)",
    }


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d.get("bf16_tflops_sustained", 1409.2), d.get("hbm_gbs", 6569.0), "measured"
    return 1400.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i",
                                          str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port of the reference algorithm on the host cores
#
# Layouts timed (BASELINE.md 4.3): (a) ONE process with torch intra-op threads = t; (b) GTSfM's own layout, a pool of worker
# PROCESSES with t threads each (gtsfm/runner.py:153-155: num_workers x threads_per_worker), every worker matching pairs
# independently.  The faster is reported; `cores` = workers x t actually busy.
# ------------------------------------------------------------------------------------------------------------------
_W = {}  # per-worker state of the process pool


def _worker_init(wname: str, threads: int):
    import cv2
    import torch

    torch.set_num_threads(threads)
    cv2.setNumThreads(threads)
    from gtsfm_b200 import synthetic as syn
    from oracle import superpoint_ref

    w = WORKLOADS[wname]
    frames, cal = syn.synthetic_sequence(4, w["H"], w["W"])
    sp_sd = syn.superpoint_state_dict(0)
    _W.update(w=w, frames=frames, cal=cal, sp_sd=sp_sd)
    if w["matcher"] == "lightglue":
        _W["m_sd"] = syn.lightglue_state_dict(2, w["profile"])
    elif w["matcher"] == "superglue":
        _W["m_sd"] = syn.superglue_state_dict(1, w["profile"])
    if w["matcher"]:
        _W["fa"] = superpoint_ref.detect_and_describe(frames[0], sp_sd, w["max_kp"])
        _W["fb"] = superpoint_ref.detect_and_describe(frames[2], sp_sd, w["max_kp"])


def _worker_task(kind: str):
    """one unit of CPU work; returns (kind, seconds)"""
    from oracle import lightglue_ref, superglue_ref, superpoint_ref, verifier_ref

    w = _W["w"]
    t0 = time.perf_counter()
    if kind == "detect":
        superpoint_ref.detect_and_describe(_W["frames"][1], _W["sp_sd"], w["max_kp"])
    else:  # one pair: match + verify
        fa, fb = _W["fa"], _W["fb"]
        shape = (w["H"], w["W"], 3)
        if w["matcher"] == "lightglue":
            m = lightglue_ref.lightglue_match(fa[0], fa[2], fb[0], fb[2], _W["m_sd"])
        else:
            m = superglue_ref.superglue_match(fa[0], fa[1], fa[2], fb[0], fb[1], fb[2], shape, shape, _W["m_sd"])
        if w["verify"]:
            verifier_ref.verify_cv2(fa[0].astype(np.float64), fb[0].astype(np.float64), m.astype(np.uint32), _W["cal"], _W["cal"], True, THR_PX)
    return kind, time.perf_counter() - t0


def cpu_layout_rate(wname: str, workers: int, threads: int, units_per_worker: int = 1):
    """Throughput of `workers` processes x `threads` threads on this workload -> (units per second of the metric, stage dict)."""
    import multiprocessing as mp

    w = WORKLOADS[wname]
    kinds = ["detect"] if not w["matcher"] else ["pair", "detect"]
    stages = {}
    if workers == 1:
        _worker_init(wname, threads)
        run = lambda kind, n: [_worker_task(kind) for _ in range(n)]  # noqa: E731
        pool = None
    else:
        pool = mp.get_context("spawn").Pool(workers, initializer=_worker_init, initargs=(wname, threads))
        run = lambda kind, n: pool.map(_worker_task, [kind] * n, chunksize=1)  # noqa: E731
    try:
        for kind in kinds:
            warm = run(kind, workers)  # warm-up (imports, first touch) outside the timed span; also sizes the sample: >= ~3 s per stage
            t_unit = max(1e-3, float(np.mean([r[1] for r in warm])))
            n = workers * max(units_per_worker, min(8, int(np.ceil(3.0 / t_unit))))
            t0 = time.perf_counter()
            res = run(kind, n)
            wall = time.perf_counter() - t0
            stages[f"{kind}_per_sec"] = n / wall
            stages[f"{kind}_s_each"] = float(np.mean([r[1] for r in res]))
    finally:
        if pool is not None:
            pool.close()
            pool.join()
    if not w["matcher"]:
        return stages["detect_per_sec"], stages
    # one detection serves `lookahead` pairs; detection and matching share the same cores
    per_pair = 1.0 / stages["pair_per_sec"] + (1.0 / stages["detect_per_sec"]) / max(1, w["lookahead"])
    return 1.0 / per_pair, stages


def cpu_baseline(wname: str, quick: bool):
    """Best CPU layout for this workload.  quick (the default CUDA run's `cpu_baseline` leg): two layouts, ~20-30 s; otherwise
    (`--impl reference`) the fuller sweep."""
    cores = os.cpu_count() or 1
    if quick:
        layouts = [(1, min(32, cores)), (max(1, cores // 8), 8)] if cores >= 16 else [(1, cores)]
    else:
        layouts = [(1, min(32, cores)), (1, min(64, cores))]
        layouts += [(max(1, cores // t), t) for t in (16, 8, 4) if cores // t >= 2]
    best = None
    tried = []
    for workers, threads in layouts:
        try:
            v, stages = cpu_layout_rate(wname, workers, threads)
        except Exception as e:  # a layout that cannot run (memory) must not sink the line
            tried.append({"workers": workers, "threads": threads, "error": repr(e)[:120]})
            continue
        tried.append({"workers": workers, "threads": threads, "value": v})
        if best is None or v > best[0]:
            best = (v, workers, threads, stages)
    v, workers, threads, stages = best
    w = WORKLOADS[wname]
    unit = "images/s" if not w["matcher"] else "pairs/s"
    sample = (f"oracle port (torch-CPU fp32 + cv2 USAC) on the host cores; layout = {workers} process(es) x {threads} threads (best of "
              f"{[(t['workers'], t['threads']) for t in tried]}); per layout: every worker runs 1 pair (match+verify at "
              f"{w['max_kp']} keypoints) and 1 detection, timed wall-clock across the pool; "
              + ("images/s = detections/s" if not w["matcher"] else f"pairs/s = 1 / (1/pair_rate + (1/detect_rate)/{max(1, w['lookahead'])})"))
    return {"value": v, "unit": unit, "cores": workers * threads, "host_cores": cores, "kind": "port", "layout": {"processes": workers, "threads_each": threads},
            "sample": sample, "stages": stages, "layouts_tried": tried}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    vals, cb = [], None
    for i in range(args.steps):  # each "step" is one bounded sweep of the layouts (tens of seconds)
        cb = cpu_baseline(args.workload, quick=False)
        vals.append(cb["value"])
    value = float(np.mean(vals))
    cb["value"] = value
    line = {
        "impl": "reference", "metric": "images_per_sec" if not w["matcher"] else "image_pairs_per_sec", "value": value, "unit": cb["unit"],
        "n_gpus": args.gpus, "steps": len(vals), "warmup": 0, "ms_per_step": 1000.0 / value, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_of(args.workload), "cpu_baseline": cb,
        "e2e": {"value": value, "unit": cb["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# CUDA arm
# ------------------------------------------------------------------------------------------------------------------
def _setup_dist():
    import torch
    import torch.distributed as dist

    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    return rank, world, local, dev


def _broadcast_weights(sds, world, dev):
    """rank 0 materialises the weights, one NCCL broadcast per model at start-up (SURVEY.md 8e)"""
    import torch
    import torch.distributed as dist

    if world == 1:
        return
    for sd, order in sds:
        blob = torch.from_numpy(np.concatenate([np.asarray(sd[k], np.float32).ravel() for k in order])).to(dev)
        dist.broadcast(blob, 0)
        flat, off = blob.cpu().numpy(), 0
        for k in order:
            n = int(np.prod(sd[k].shape)) if sd[k].shape else 1
            sd[k] = flat[off:off + n].reshape(sd[k].shape)
            off += n


DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this much


def dump_outputs(out: Path, step: dict) -> None:
    """Write what the last timed step returned to its caller, as .npy files under `out` (float32, or float64 where a float32
    could not hold every value exactly):
      keypoints (N, 2), scores (N,), keypoints_per_frame (F,)   the step's new frames, concatenated in frame order
      descriptors (D, 256), descriptor_rows (D,)                 the rows of the concatenated descriptors: all N, or a fixed seeded
                                                                 sample of them where all would not fit in DUMP_BYTES
      matches (M, 2), matches_per_pair (P,), stop_layer (P,)     pairs ordered by (new frame, window slot); stop_layer for LightGlue
      inlier_mask (M,), num_inliers (P,), essential (P, 3, 3), rotation (P, 3, 3), translation (P, 3)
                                                                 each pair's verification; NaN where it found no model"""
    import torch

    feats = step["features"]
    arrays = {"keypoints": torch.cat([f.kp for f in feats]).float().cpu().numpy(),
              "scores": torch.cat([f.score for f in feats]).float().cpu().numpy(),
              "keypoints_per_frame": np.array([len(f) for f in feats], np.float64)}
    pairs = [step["pairs"][k] for k in sorted(step.get("pairs", {}))]
    if pairs:
        arrays["matches"] = np.concatenate([p["matches"].cpu().numpy().reshape(-1, 2) for p in pairs]).astype(np.float64)
        arrays["matches_per_pair"] = np.array([p["matches"].shape[0] for p in pairs], np.float64)
        if "stop" in pairs[0]:
            arrays["stop_layer"] = np.array([p["stop"] for p in pairs], np.float64)
        nan = lambda shape: np.full(shape, np.nan)  # noqa: E731
        verified = [p["verify"] for p in pairs]
        arrays["inlier_mask"] = np.concatenate([v[4].cpu().numpy() for v in verified]).astype(np.float32)
        arrays["num_inliers"] = np.array([v[3] for v in verified], np.float64)
        arrays["essential"] = np.stack([nan((3, 3)) if v[0] is None else v[0] for v in verified]).astype(np.float64)
        arrays["rotation"] = np.stack([nan((3, 3)) if v[1] is None else v[1] for v in verified]).astype(np.float64)
        arrays["translation"] = np.stack([nan(3) if v[2] is None else np.asarray(v[2]).ravel() for v in verified]).astype(np.float64)
    n = int(arrays["keypoints"].shape[0])
    fit = (DUMP_BYTES - 4096 - sum(a.nbytes for a in arrays.values())) // (256 * 4 + 8)  # 4096: room for the .npy headers
    rows = np.arange(n) if n <= fit else np.sort(np.random.default_rng(0).choice(n, fit, replace=False))
    desc = torch.cat([f.desc for f in feats])
    arrays["descriptors"] = desc[torch.from_numpy(rows).to(desc.device)].float().cpu().numpy()
    arrays["descriptor_rows"] = rows.astype(np.float64)
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_BYTES
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a)


def run_cuda(args):
    import torch
    import torch.distributed as dist

    from gtsfm_b200 import synthetic as syn, weights
    from gtsfm_b200.detector_descriptor import B200SuperPointDetectorDescriptor
    from gtsfm_b200.gtsfm_api import Cal3Bundler, Image
    from gtsfm_b200.matcher import B200LightGlueMatcher, B200SuperGlueMatcher
    from gtsfm_b200.pipeline import DeviceFrontEnd
    from gtsfm_b200.verifier import B200Ransac

    wname = args.workload
    w = WORKLOADS[wname]
    H, W, MAX_KP, LOOKAHEAD, NEW_FRAMES = w["H"], w["W"], w["max_kp"], w["lookahead"], w["new_frames"]
    units_per_step = NEW_FRAMES if not w["matcher"] else LOOKAHEAD * NEW_FRAMES
    rank, world, local, dev = _setup_dist()
    sp_sd = syn.superpoint_state_dict(0)
    lg_sd = syn.lightglue_state_dict(2, w["profile"]) if w["matcher"] == "lightglue" else None
    sg_sd = syn.superglue_state_dict(1, w["profile"]) if w["matcher"] == "superglue" else None
    sds = [(sp_sd, weights.SUPERPOINT_ORDER)]
    if lg_sd is not None:
        sds.append((lg_sd, weights.LIGHTGLUE_ORDER))
    _broadcast_weights(sds, world, dev)
    fe = DeviceFrontEnd(sp_sd, lg_sd, device=local, max_keypoints=MAX_KP, superglue_sd=sg_sd, fp16_attention=args.fp16_attention)
    if args.lg_batch:
        fe.ctx.set_option("lightglue_batch", args.lg_batch)
    n_frames = max(LOOKAHEAD, 1) + NEW_FRAMES * (args.warmup + args.steps) * 2 + 4
    n_frames = min(n_frames, 96) if not w["matcher"] else n_frames  # detect-only: frames are re-used round robin
    # each rank works on its own stretch of the sequence (weak scaling): different seed per rank
    frames, cal = syn.synthetic_sequence(n_frames, H, W, seed=77 + rank)
    frames_dev = [torch.from_numpy(f).to(dev) for f in frames]
    torch.cuda.synchronize()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    window = deque(maxlen=max(LOOKAHEAD, 1))
    for i in range(LOOKAHEAD):
        window.append(fe.detect(frames_dev[i]))
    cursor = LOOKAHEAD
    stats = {"matches": 0, "inliers": 0, "pairs": 0, "stops": 0, "keypoints": 0, "frames": 0}

    stats_lock = threading.Lock()

    def step_device(c, record=None):
        """One step.  `record` (a dict) receives what the step hands its caller: the new frames' features in order, and per pair
        (key (new frame, window slot)) the matches, the LightGlue stop layer and the verification result."""
        pending = []
        if not w["matcher"]:  # detect-describe only: every frame of the step enqueued before the first count is read
            for f in fe.detect_many([frames_dev[(c + j) % len(frames_dev)] for j in range(NEW_FRAMES)]):
                stats["keypoints"] += len(f)
                stats["frames"] += 1
                if record is not None:
                    record.setdefault("features", []).append(f)
            return
        for j in range(NEW_FRAMES):
            f = fe.detect(frames_dev[(c + j) % len(frames_dev)])
            stats["keypoints"] += len(f)
            stats["frames"] += 1
            if record is not None:
                record.setdefault("features", []).append(f)
            if not w["matcher"]:
                continue
            prevs = list(window)
            if w["matcher"] == "lightglue":
                # lock-step batches of 8 pairs (b2_lightglue_match_batched_dev) over MATCH_LANES concurrent LightGlue instances;
                # a batch's verifications are queued the moment it completes and overlap the other batches' matcher kernels
                def on_chunk(c0, res, prevs=prevs, f=f, j=j):
                    with stats_lock:
                        for i, (prev, (m, stop)) in enumerate(zip(prevs[c0:c0 + len(res)], res)):
                            pending.append(((j, c0 + i), fe.verify_async(prev, f, m, cal, cal, THR_PX)))
                            stats["matches"] += int(m.shape[0])
                            stats["stops"] += stop
                            stats["pairs"] += 1
                            if record is not None:
                                record.setdefault("pairs", {})[(j, c0 + i)] = {"matches": m, "stop": stop}

                fe.match_many([(prev, f) for prev in prevs], on_chunk=on_chunk)
            else:
                def on_pair(i, m, prevs=prevs, f=f, j=j):  # a pair's verification is queued the moment its matches exist
                    with stats_lock:
                        pending.append(((j, i), fe.verify_async(prevs[i], f, m, cal, cal, THR_PX)))
                        stats["matches"] += int(m.shape[0])
                        stats["pairs"] += 1
                        if record is not None:
                            record.setdefault("pairs", {})[(j, i)] = {"matches": m}

                fe.match_superglue_many([(prev, f) for prev in prevs], on_pair=on_pair)
            window.append(f)
        for key, fut in pending:  # every verification result is collected inside the step
            res = fut.result()
            stats["inliers"] += res[3]
            if record is not None:
                record["pairs"][key]["verify"] = res

    for _ in range(args.warmup):
        step_device(cursor)
        cursor += NEW_FRAMES
    for k in stats:
        stats[k] = 0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    launches0 = fe.launch_count()
    vlaunch0 = fe._vctx.launch_count() if fe._vctx else 0
    # With B2_SP_GRAPH=1 the SuperPoint network is replayed as ONE CUDA graph per image; per-launch CUDA events cannot see inside
    # a graph (the library launches directly while a kernel of the network is being profiled).  Then, when the dominant kernel
    # lives inside that graph (superpoint_only), the timed pass runs unprofiled and the kernel is timed in a second pass over the
    # same number of steps.  Default (graph off): the dominant kernel is timed live inside the timed pass.
    in_graph = os.environ.get("B2_SP_GRAPH") == "1" and w["dominant"].startswith(("k_conv", "k_nms", "k_head"))

    def timed_pass(c, record=None):
        tot = 0.0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for s in range(args.steps):
            flush.fill_(1)  # L2 flush, outside the timed span
            torch.cuda.synchronize()
            e0.record()
            step_device(c, record if s == args.steps - 1 else None)
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
            c += NEW_FRAMES
        return tot, c

    if not in_graph:
        fe.profile_start(w["dominant"])
    last_step = {} if args.dump_outputs and rank == 0 else None
    total_ms, cursor = timed_pass(cursor, last_step)
    if not in_graph:
        k_ms, k_launches, k_work = fe.profile_stop()
        prof_total_ms = total_ms
    if last_step is not None:  # before any later step can reuse the matcher's output buffers
        dump_outputs(Path(args.dump_outputs), last_step)
    launches = fe.launch_count() - launches0 + (fe._vctx.launch_count() - vlaunch0 if fe._vctx else 0)
    if in_graph:
        keep = dict(stats)
        fe.profile_start(w["dominant"])
        prof_total_ms, cursor = timed_pass(cursor)
        k_ms, k_launches, k_work = fe.profile_stop()
        stats.update(keep)
    # secondary figures (untimed region): where the rest of the step goes - one extra step per kernel family, CUDA events around
    # every launch of that family on its launching stream (the verification kernels run on their own context / stream)
    family_ms = {}
    if w["matcher"]:
        for fam in ("k_gemm_ws", "k_lg_", "k_sg_", "k_conv", "k_nms", "k_head"):
            fe.profile_start(fam)
            step_device(cursor)
            torch.cuda.synchronize()
            ms, n, _ = fe.profile_stop()
            if n:
                family_ms[fam] = {"ms_per_step": ms, "launches": n}
        if fe._vctx is not None:
            fe._vctx.profile_start("k_rs_")
            step_device(cursor)
            torch.cuda.synchronize()
            ms, n, _ = fe._vctx.profile_stop()
            family_ms["k_rs_ (verification stream, overlapped)"] = {"ms_per_step": ms, "launches": n}
    # detect-only rate (BASELINE configs[1] shape) and the encoder convolutions' rate
    torch.cuda.synchronize()
    fe.ctx.profile_start("k_conv_ps")
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0.record()
    for j in range(16):
        fe.detect(frames_dev[j % len(frames_dev)])
    d1.record()
    torch.cuda.synchronize()
    conv_ms, conv_n, conv_flop = fe.ctx.profile_stop()
    detect_ips = 16.0 / (d0.elapsed_time(d1) / 1e3)
    barrier()
    clocks = sampler.stop()
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    max_ms = float(t.item())
    units_total = units_per_step * args.steps * world
    value = units_total / (max_ms / 1000.0)

    # ---- e2e: the same step through the GTSfM plugin API with host buffers ------------------------------------------
    det = B200SuperPointDetectorDescriptor(max_keypoints=MAX_KP, weights_path=sp_sd, device=local)
    calib = Cal3Bundler(cal[0], 0, 0, cal[1], cal[2])

    def make_matcher(cache: bool):
        if w["matcher"] == "lightglue":
            return B200LightGlueMatcher("superpoint", weights_path=lg_sd, device=local, feature_cache=cache)
        if w["matcher"] == "superglue":
            return B200SuperGlueMatcher(weights_path=sg_sd, device=local)
        return None

    def e2e_run(cache: bool, steps: int, nthreads: int = 1):
        """The step through the plugin classes with HOST buffers.  nthreads > 1: the step's plugin calls are issued from a pool
        of host threads, each with its OWN plugin instances (own library context / stream), the way a GTSfM deployment issues
        them from several Dask worker threads - one pair's copies, per-layer host syncs and latency-bound RANSAC kernels then
        overlap another pair's matching on the GPU.  Same calls, same work, same host-in / host-out contract."""
        import concurrent.futures as cf

        tls = threading.local()
        made, lock = [], threading.Lock()

        def state():
            if not hasattr(tls, "st"):
                st = {"mat": make_matcher(cache), "ver": B200Ransac(True, THR_PX, device=local) if w["verify"] else None,
                      "det": None if w["matcher"] else B200SuperPointDetectorDescriptor(max_keypoints=MAX_KP, weights_path=sp_sd, device=local)}
                tls.st = st
                with lock:
                    made.append(st)
            return tls.st

        def do_pair(task):
            pk, pd, kps, desc = task
            st = state()
            m = st["mat"].match(pk, kps, pd, desc, (H, W, 3), (H, W, 3))
            if st["ver"] is not None:
                st["ver"].verify(pk, kps, m, calib, calib)

        def do_frame(idx):
            state()["det"].detect_and_describe(Image(frames[idx % len(frames)]))

        pool = cf.ThreadPoolExecutor(nthreads) if nthreads > 1 else None
        run = (lambda fn, items: list(pool.map(fn, items))) if pool else (lambda fn, items: [fn(x) for x in items])
        hwin = deque(maxlen=max(LOOKAHEAD, 1))
        for i in range(LOOKAHEAD):
            hwin.append(det.detect_and_describe(Image(frames[i])))

        def step_host(c):
            if not w["matcher"]:
                run(do_frame, [c + j for j in range(NEW_FRAMES)])
                return
            for j in range(NEW_FRAMES):
                kps, desc = det.detect_and_describe(Image(frames[(c + j) % len(frames)]))
                run(do_pair, [(pk, pd, kps, desc) for pk, pd in list(hwin)])
                hwin.append((kps, desc))

        def copied():
            engs = [det._engine]
            for st in made:
                engs += [st["mat"]._engine if st["mat"] else None, st["ver"]._engine if st["ver"] else None, st["det"]._engine if st["det"] else None]
            return sum(e.h2d_bytes for e in engs if e), sum(e.d2h_bytes for e in engs if e)

        c2 = LOOKAHEAD
        for _ in range(min(args.warmup, 2)):
            step_host(c2)
            c2 += NEW_FRAMES
        barrier()
        h2d0, d2h0 = copied()
        wall = 0.0
        for _ in range(steps):
            flush.fill_(1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            step_host(c2)
            torch.cuda.synchronize()
            wall += time.perf_counter() - t0
            c2 += NEW_FRAMES
        barrier()
        if pool:
            pool.shutdown()
        tt = torch.tensor([wall], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        h2d1, d2h1 = copied()
        return units_per_step * steps * world / float(tt.item()), (h2d1 - h2d0) // steps, (d2h1 - d2h0) // steps

    if args.no_e2e:
        e2e_value, h2d, d2h = float("nan"), 0, 0
    else:
        e2e_value, h2d, d2h = e2e_run(False, args.steps, args.e2e_threads)
    e2e = {"value": e2e_value, "unit": "images/s" if not w["matcher"] else "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "host_threads": args.e2e_threads,
           "host_threads_note": "plugin calls issued from this many host threads, each with its own plugin instances (what Dask worker threads do); "
                                "single_thread = the same loop from one thread",
           "feature_cache": "off (default: every call uploads its arrays, like the reference)"}
    if not args.no_e2e and args.e2e_threads > 1:
        e2e["single_thread"] = e2e_run(False, max(1, args.steps - 1), 1)[0]
    if w["matcher"] == "lightglue" and not args.no_e2e:
        v2, h2, _ = e2e_run(True, max(1, args.steps - 1))
        e2e["with_feature_cache"] = {"value": v2, "h2d_bytes_per_step": int(h2), "note": "opt-in B200LightGlueMatcher(feature_cache=True), full-content hash"}

    if rank == 0:
        tf_peak, hbm_peak, peak_src = measured_peaks()
        achieved = (k_work / 1e12) / (k_ms / 1e3) if k_ms > 0 else 0.0
        unit = "images/s" if not w["matcher"] else "pairs/s"
        line = {
            "metric": "images_per_sec" if not w["matcher"] else "image_pairs_per_sec", "value": value, "unit": unit, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": max_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config_of(wname), "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": w["dominant"], "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s",
                         "frac": achieved / tf_peak, "traffic": DOMINANT_DRAM_BYTES.get(wname),
                         "traffic_unit": "dram__bytes_read.sum + dram__bytes_write.sum of one launch (ncu --set full capture under profiles/, the launch shape named in bench.py DOMINANT_DRAM_BYTES); null = no capture of this workload's launch shape",
                         "peak_source": f"bf16_tflops_sustained ({peak_src})",
                         "kernel_ms_per_step": k_ms / args.steps, "kernel_launches_per_step": k_launches / args.steps,
                         "kernel_share_of_step": k_ms / prof_total_ms if prof_total_ms else None,
                         "kernel_timing": ("second pass of the same steps with direct launches (the timed pass replays the network as a CUDA graph, "
                                           f"which per-launch events cannot see); that pass took {prof_total_ms / args.steps:.2f} ms per step") if in_graph
                         else ("CUDA events around every launch inside the timed pass" +
                               (f"; {DETECT_LANES} SuperPoint lanes run concurrently, so a launch shares the SMs with other lanes' kernels and "
                                "the summed kernel time exceeds the step time (the kernel alone: profiles/r02_conv_ps_*.txt)"
                                if not w["matcher"] and DETECT_LANES > 1 else
                                "; 3 SuperGlue instances match pairs concurrently (match_superglue_many), so a launch shares the SMs with the other "
                                "lanes' kernels: per-launch time, and with it this fraction, is inflated by the contention (one lane: 0.24)"
                                if w["matcher"] == "superglue" else "")),
                         "note": "split-fp16 x3 products: tensor-pipe FLOPs are 3x the algorithmic FLOPs counted here (ceiling of frac = 0.33)"},
            "work": {"matches_per_pair": stats["matches"] / max(1, stats["pairs"]), "inliers_per_pair": stats["inliers"] / max(1, stats["pairs"]),
                     "mean_stop_layer": stats["stops"] / max(1, stats["pairs"]) if w["matcher"] == "lightglue" else None,
                     "keypoints_per_frame": stats["keypoints"] / max(1, stats["frames"])},
            "encoder_conv_frac": ((conv_flop / 1e12) / (conv_ms / 1e3)) / tf_peak if conv_ms > 0 else None,
            "extra": {"superpoint_detect_describe_images_per_sec_1gpu": detect_ips,
                      "encoder_conv_tflops": (conv_flop / 1e12) / (conv_ms / 1e3) if conv_ms > 0 else None,
                      "kernel_family_ms_per_step": family_ms},
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(wname, quick=True)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_strong(args):
    """One fixed job through the real L2 seam: F frames, Sequential(lookahead 20) pairs, B200CorrespondenceGenerator (every image
    detected on one rank and its features all-gathered over NCCL, every rank matches its p mod world shard in batches of 8 with each batch's two-view verification queued
    on the verification stream as it completes, all_gather_object of the match arrays).  Wall-clock on rank 0 between two barriers; total work is fixed => "strong"."""
    import torch
    import torch.distributed as dist

    from gtsfm_b200 import distributed as D, synthetic as syn
    from gtsfm_b200.correspondence_generator import B200CorrespondenceGenerator
    from gtsfm_b200.gtsfm_api import Image

    rank, world, local, dev = _setup_dist()
    F, L = args.frames, 20
    frames, cal = syn.synthetic_sequence(F, 480, 640, seed=77)
    images = [Image(f) for f in frames]
    graph = [(i, j) for i in range(F) for j in range(i + 1, min(F, i + L + 1))]  # sequential_retriever.py:57-59
    gen = B200CorrespondenceGenerator(syn.superpoint_state_dict(0), syn.lightglue_state_dict(2, "bench"), max_keypoints=5000, device=local)
    warm = [(i, j) for i in range(6) for j in range(i + 1, 6)]  # warm-up: contexts, 8-pair workspaces, verification lane, NCCL
    gen.generate_correspondences(None, images[:6], warm, verify_with=({i: cal for i in range(6)}, THR_PX))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    wall = t_corr = 0.0
    for _ in range(args.steps):  # one step = the whole job
        barrier()
        t0 = time.perf_counter()
        kps, matches = gen.generate_correspondences(None, images, graph, verify_with=({i: cal for i in range(F)}, THR_PX))
        t_corr += time.perf_counter() - t0
        fe = gen._front_end()
        feats = gen.last_device_features
        res = gen.last_two_view  # this rank's shard, verified under the matching (B200TwoViewBatch semantics)
        n_ok = sum(1 for r in res.values() if r.i2Ri1 is not None)
        barrier()
        wall += time.perf_counter() - t0
    wall, t_corr = wall / args.steps, t_corr / args.steps  # per job
    tt = torch.tensor([wall, t_corr, float(gen.last_detections), float(n_ok)], dtype=torch.float64, device=dev)
    if world > 1:
        mx = tt.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = tt.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        wall, t_corr, det_total, ok_total = float(mx[0]), float(mx[1]), float(sm[2]), float(sm[3])
    else:
        det_total, ok_total = float(gen.last_detections), float(n_ok)
    if rank == 0:
        cfg = config_of("vga_lightglue")
        cfg["workload"] = (f"strong scaling: ONE job of {F} synthetic 640x480 frames, Sequential lookahead 20 = {len(graph)} pairs (BASELINE configs[3] shape; "
                           f"F = 500 gives its 9 790-pair graph), B200CorrespondenceGenerator with the two-view verification run under the matching, pairs sharded p mod world")
        line = {
            "metric": "image_pairs_per_sec", "value": len(graph) / wall, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": 1,
            "ms_per_step": wall * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "gpu_launches": int(fe.launch_count()),
            "strong": {"pairs": len(graph), "frames": F, "wall_s": wall, "correspondence_s_max_rank": t_corr,
                       "phases_rank0_s": gen.last_timing, "detections_summed_over_ranks": det_total, "detections_if_not_duplicated": F, "verified_pairs": ok_total,
                       "exchange": "each image detected on one rank (position mod world), features all-gathered over NCCL once; matches "
                                   "all_gather_object'ed at the end",
                       "limits": "what does not shrink with the number of GPUs: the feature all-gather (5 MB per image to every rank), the final "
                                 "all_gather_object that pickles every (K, 2) match array to every rank, host-side result conversion"},
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default="vga_lightglue", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--frames", type=int, default=120, help="--scaling strong: frames of the fixed job (500 = BASELINE configs[3])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-threads", type=int, default=4, help="host threads issuing the plugin calls of the e2e leg (each with its own plugin instances)")
    ap.add_argument("--no-e2e", action="store_true", help="experiments only: skip the plugin-path leg (the line is then not a valid bench line)")
    ap.add_argument("--fp16-attention", action="store_true",
                    help="opt-in mode: the reference's CUDA numerics for attention (fp16 flash SDPA, one MMA per product); NOT the "
                         "parity-pinned default - the line says so in config.matcher")
    ap.add_argument("--lg-batch", type=int, default=0, help="experiments: pairs per lock-step LightGlue batch inside the library (0 = default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "cuda" or args.scaling != "weak"):
        ap.error("--dump-outputs applies to the CUDA arm's weak-scaling steps")
    global FP16_ATTN
    FP16_ATTN = bool(args.fp16_attention)
    if args.impl == "reference":
        run_reference(args)
    elif args.scaling == "strong":
        run_strong(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
