#!/usr/bin/env python
"""bench.py -- end-to-end frames/s of the per-frame ADAS path (YOLOv8l + UFLDv2-CULane-ResNet34 + ByteTrack) on
synthetic 1280x720 frames, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch 8] [--impl b200|reference] [--dump-outputs DIR]

A "step" = one batch of `--batch` consecutive frames of one stream through the whole hot path:
    frames -> [letterbox + YOLOv8l + DFL decode + candidate select + reference NMS]  (adas_yolo_detect)
           -> [resize/crop/normalise + UFLDv2-res34 + row/col-anchor decode]         (adas_ufld_detect)
           -> ByteTrack update per frame, in order (device IoU-cost + LAP kernels)   (BYTETracker.update)
`value`  : frames already resident in HBM (device pointers), timed with CUDA events on the engines' own streams.
`e2e`    : the same steps fed from pinned HOST memory through the reference-facing API (H2D inside the timed region,
           results read back to the host every step) -- the headline number.
`--impl reference` times the oracle's CPU port of the reference path (reference Python semantics, torch-CPU fp32
nets with the same seeded weights; onnxruntime is not installed, so ORT-CPU is substituted by torch-CPU) on a
bounded sample.  Multi-GPU (torchrun): every rank runs its own stream (weak scaling); the only collective is an
NCCL all_gather of the fixed-size detection records per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FRAME_H, FRAME_W = 720, 1280
BOX_SCORE, NMS_IOU, MAX_DET = 0.4, 0.45, 300


def synth_stream(seed: int, n: int) -> np.ndarray:
    """n frames of a moving-rectangles scene over noise (SURVEY 8d synthetic inputs), uint8 BGR."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (FRAME_H, FRAME_W, 3), dtype=np.uint8)
    k = 24
    pos = rng.uniform(0, 1, (k, 2)) * (FRAME_W - 200, FRAME_H - 200)
    vel = rng.uniform(-6, 6, (k, 2))
    size = rng.integers(40, 260, (k, 2))
    col = rng.integers(0, 256, (k, 3), dtype=np.uint8)
    out = np.empty((n, FRAME_H, FRAME_W, 3), np.uint8)
    for f in range(n):
        img = base.copy()
        for j in range(k):
            x, y = (pos[j] + vel[j] * f).astype(int)
            x, y = int(np.clip(x, 0, FRAME_W - 10)), int(np.clip(y, 0, FRAME_H - 10))
            img[y:y + size[j, 1], x:x + size[j, 0]] = col[j]
        out[f] = img
    return out


def build_plans(seed: int = 0):
    import adas_b200  # noqa: F401
    from adas_b200 import plan
    CACHE = plan.cache_dir()
    out = {}
    for kind, builder, kw in (("yolov8", plan.build_yolov8, dict(scale="l")), ("ufldv2", plan.build_ufldv2, dict(backbone="34"))):
        import zlib
        prof = zlib.crc32(repr((plan.SYNTH_PROFILES.get(kind), plan.SYNTH_PROFILES_WORKLOAD.get(kind), plan.PLAN_VERSION)).encode()) & 0xffff
        path = os.path.join(CACHE, f"bench_{kind}_s{seed}_workload_{prof:04x}.b200w")
        W = plan.synth_weights(kind, seed, variant=kw.get("scale", kw.get("backbone")), workload=True)
        pb = builder(W, **kw)
        if not os.path.isfile(path):
            pb.write(path + f".{os.getpid()}.tmp")
            os.replace(path + f".{os.getpid()}.tmp", path)
        out[kind] = (path, W.state_dict, pb)
    return out


DUMP_LIMIT = 64 << 20


def _step_arrays(r, frames) -> dict:
    f = np.asarray(frames)
    counts, npts = np.asarray(r.counts)[f], np.asarray(r.lane_npts)[f]
    det = np.arange(r.boxes.shape[1])[None, :] < counts[:, None]                   # [F, max_det]: rows past the count are unset
    pts = np.arange(r.lane_pts.shape[2])[None, None, :] < npts[:, :, None]        # [F, 4, max_pts]
    recs = [r.tracks[i] for i in f.tolist()]
    cols = [np.concatenate([t[n].reshape(len(t), int(np.prod(t.dtype[n].shape))).astype(np.float64) for n in t.dtype.names], 1)
            for t in recs]
    return {
        "frame_index": f.astype(np.float64),
        "det_boxes": np.where(det[..., None], r.boxes[f], 0).astype(np.float32),
        "det_scores": np.where(det, r.scores[f], 0).astype(np.float32),
        "det_class_ids": np.where(det, r.class_ids[f], -1).astype(np.float64),
        "det_cand_index": np.where(det, r.cand_index[f], -1).astype(np.float64),
        "det_counts": counts.astype(np.float64),
        "det_n_candidates": np.asarray(r.n_candidates)[f].astype(np.float64),
        "lane_pts": np.where(pts[..., None], r.lane_pts[f], 0).astype(np.float64),
        "lane_npts": npts.astype(np.float64),
        "lane_status": np.asarray(r.lane_status)[f].astype(np.float64),
        "track_counts": np.array([len(t) for t in recs], np.float64),
        "tracks": np.concatenate(cols),
    }


def dump_outputs(r, out_dir: str, limit: int = DUMP_LIMIT) -> dict:
    """Write what one pipeline step handed its caller as out_dir/<name>.npy (float32 / float64) so that two builds can be
    compared output for output: detections (xywh boxes, scores, class ids, candidate indices, per-frame counts), lanes (points,
    counts, status) and the tracker's records of every frame, concatenated in frame order (`track_counts` rows per frame; columns
    are the fields of adas_b200._capi.TRACK_DTYPE in order, arrays flattened).  Entries past a frame's count hold no result and are
    written as zeros (-1 for ids), so equal inputs give equal files.  If the batch would exceed `limit` bytes, a fixed, seeded
    sample of its frames is written instead; `frame_index` lists the frames kept."""
    B = int(np.asarray(r.counts).shape[0])
    keep = np.arange(B)
    arrays = _step_arrays(r, keep)
    size = sum(a.nbytes for a in arrays.values())
    while size > limit and len(keep) > 1:
        n = max(1, min(len(keep) - 1, len(keep) * limit // size))
        keep = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
        arrays = _step_arrays(r, keep)
        size = sum(a.nbytes for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return arrays


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line).  One nvidia-smi process
    logs every 25 ms for the whole run (its start-up takes longer than a short timed region); each line carries nvidia-smi's own
    timestamp and `window(t0, t1)` keeps the samples taken between the two wall-clock marks of a timed region."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            t_end = time.time() + 3.0
            while not self.lines and time.time() < t_end:      # first sample = the logger is up
                time.sleep(0.02)
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    @staticmethod
    def _stamp(txt: str, arrival: float) -> float:
        import datetime
        try:
            return datetime.datetime.strptime(txt.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return arrival

    def window(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.05)                                        # let the samples of the last few ms arrive
        sm, mx, reasons = [], [], set()
        for arrival, ln in list(self.lines):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 10:
                continue
            ts = self._stamp(f[0], arrival)
            if ts < t0 - 0.002 or ts > t1 + 0.002:
                continue
            try:
                sm.append(float(f[2])); mx.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[6:10]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}

    def close(self):
        if self.proc is not None:
            self.proc.terminate()


# ------------------------------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    import adas_b200  # noqa: F401
    from adas_b200 import _capi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"        # keep stdout to the one JSON line (NCCL prints its version banner there)
        # NCCL prints its version banner on stdout when the first communicator is created: keep stdout to the one JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    B, K, Wm = args.batch, args.steps, max(args.warmup, 3)
    if rank == 0:
        plans = build_plans()
    if world > 1:
        dist.barrier()
    if rank != 0:
        plans = build_plans()
    from adas_b200.pipeline import AdasPipeline
    pipe = AdasPipeline(plans["yolov8"][0], plans["ufldv2"][0], device=local, batch=B, box_score=BOX_SCORE, box_nms_iou=NMS_IOU, max_det=MAX_DET,
                        sets=args.sets, depth=args.depth)

    # one stream per rank; frames differ per step (pool larger than L2: 24 batches x 22 MB = 530 MB >> 126 MB)
    pool_batches = max(6, min(24, 192 // B))
    stream = synth_stream(1000 + rank, B * 4)
    host_pool = torch.empty((pool_batches, B, FRAME_H, FRAME_W, 3), dtype=torch.uint8).pin_memory()
    hp = host_pool.numpy()
    for i in range(pool_batches):
        hp[i] = np.roll(stream[(i % 4) * B:(i % 4 + 1) * B], shift=3 * i, axis=2)
    dev_pool = host_pool.to(f"cuda:{local}")
    torch.cuda.synchronize()
    # BASELINE configs[4] "NCCL gather of boxes": EVERY batch's detection / track records ([B, 300, 7] fp32, 67 KB) are all-gathered
    # across the ranks inside the timed region: one library call per step (adas_comm_all_gather) stages the block, uploads it and runs
    # ncclAllGather on the library's private stream with its own communicator -- no torch.distributed and no host synchronisation in
    # the loop (round 1 exchanged once per run of steps because the Python-issued per-step collective cost 0.5 ms per step).
    multi = world > 1 and os.environ.get("ADAS_B200_NO_GATHER") != "1"
    comm = None
    rec = np.zeros((B, MAX_DET, 7), np.float32) if multi else None
    if multi:
        from adas_b200 import _capi as _c
        idt = torch.zeros(128, dtype=torch.uint8, device=f"cuda:{local}")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(_c.Comm.unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)                      # start-up only: hand rank 0's NCCL id to the other ranks
        sys.stdout.flush()
        saved_fd2 = os.dup(1)
        os.dup2(2, 1)                               # a new communicator may print the NCCL banner on stdout
        try:
            comm = _c.Comm(local, rank, world, bytes(idt.cpu().numpy().tobytes()), rec.nbytes)
            comm.all_gather(rec)
            comm.sync()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd2, 1)
            os.close(saved_fd2)
    gather_n = [0]

    def gather(r):
        if not multi or r is None:
            return
        gather_n[0] += 1
        rec[..., :4], rec[..., 4], rec[..., 5] = r.boxes, r.scores, r.class_ids
        rec[..., 6] = 0
        for b, tr in enumerate(r.tracks or []):
            n = min(len(tr), MAX_DET)
            if n:
                rec[b, :n, 6] = tr["track_id"][:n]
        comm.all_gather(rec)                        # asynchronous: returns as soon as the block is staged and the collective is enqueued

    def final_gather():
        if multi:
            comm.sync()                             # every step's gather has completed before the timed region closes

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    copy_stream = torch.cuda.Stream()
    NS = pipe.depth + 2            # staging slots: batches in flight + the one being uploaded
    stage = [torch.empty((B, FRAME_H, FRAME_W, 3), dtype=torch.uint8, device=f"cuda:{local}") for _ in range(NS)]
    copy_ev = [torch.cuda.Event() for _ in range(NS)]

    def upload(slot, j):            # pinned host -> device staging on a side stream (overlaps the previous batch's compute)
        with torch.cuda.stream(copy_stream):
            stage[slot].copy_(host_pool[j], non_blocking=True)
            copy_ev[slot].record(copy_stream)

    def run_steps(n, first, on_device):
        """n steps from pool batch `first` on; returns the result of the last one"""
        last = None
        if not on_device:
            upload(0, first % pool_batches)
        for i in range(n):
            j = (first + i) % pool_batches
            if on_device:
                ptr = dev_pool[j].data_ptr()
            else:
                copy_ev[i % NS].synchronize()
                if i + 1 < n:
                    upload((i + 1) % NS, (first + i + 1) % pool_batches)
                ptr = stage[i % NS].data_ptr()
            r = pipe.step_pipelined(ptr, True, (B, FRAME_H, FRAME_W))
            gather(r)
            last = r if r is not None else last
        for r in pipe.flush():
            gather(r)
            last = r
        final_gather()
        return last

    sampler = ClockSampler(local)

    def timed(on_device: bool):
        run_steps(Wm, 0, on_device)
        barrier()
        n0 = _capi.launch_count()
        w0 = time.time()
        pipe.yolo.event_record(0)
        t0 = time.perf_counter()
        last = run_steps(K, Wm, on_device)
        pipe.ufld.event_record(1)
        pipe.yolo.event_record(1)
        torch.cuda.synchronize()
        ms_dev = max(pipe.yolo.elapsed_ms(0, pipe.ufld, 1), pipe.yolo.elapsed_ms(0, pipe.yolo, 1))
        ms_wall = (time.perf_counter() - t0) * 1e3
        clocks = sampler.window(w0, time.time())
        launches = _capi.launch_count() - n0
        barrier()
        # the tracker of the last batch runs on the host after the last device event: take the larger of the two clocks
        ms = max(ms_dev, ms_wall)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{local}")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches, clocks, last

    if args.profile_steps:
        # profiler target (ncu --profile-from-start off): warm up (autotune, graph capture), then expose N steps; no numbers printed
        run_steps(Wm + 2, 0, True)
        barrier()
        torch.cuda.profiler.start()
        run_steps(args.profile_steps, Wm, True)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        pipe.close()
        return
    sampler.start()
    ms_dev, launches, clocks, _ = timed(True)
    ms_e2e, _, clocks_e2e, last = timed(False)
    sampler.close()
    if args.dump_outputs and rank == 0:
        dump_outputs(last, args.dump_outputs)

    result = None
    if rank == 0:
        fps = world * B * K / (ms_dev / 1e3)
        fps_e2e = world * B * K / (ms_e2e / 1e3)
        # roofline of the dominant kernel (conv_gemm_v3_kernel / conv_chain_v3_kernel): all GEMM launches of one step back to back on the engine stream
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("bf16_tflops", 1590.0))
        ms_y, n_y = pipe.yolo.time_ops(B, 1 << 1, 5)
        ms_u, n_u = pipe.ufld.time_ops(B, 1 << 1, 5)
        ms_all_y, _ = pipe.yolo.time_ops(B, 0xFFFFFFFF, 5)
        ms_all_u, _ = pipe.ufld.time_ops(B, 0xFFFFFFFF, 5)
        # FLOPs of the launches that are timed here: the stem convs run in stem_conv.cu (warp MMA), not in the tcgen05 GEMM launches
        gf_y = (plans["yolov8"][2].flops_per_img - plans["yolov8"][2].stem_flops_per_img) / 1e9
        gf_u = (plans["ufldv2"][2].flops_per_img - plans["ufldv2"][2].stem_flops_per_img) / 1e9
        gflop_step = (gf_y + gf_u) * B
        achieved = gflop_step / (ms_y + ms_u)          # GFLOP / ms == TFLOP/s
        # DRAM bytes per GEMM launch: measured by ncu over whole steps of THIS command (bench.py --profile-steps, caches not flushed
        # between launches); tools/traffic_report.py turns the capture into the JSON read here.  null if the capture is absent.
        traffic, traffic_detail = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "r02_bench_traffic.json")))
            if tj.get("batch") == B:
                traffic = tj.get("dram_bytes_per_launch")
                traffic_detail = {k: tj.get(k) for k in ("gemm_dram_bytes_per_step", "algorithmic_bytes_per_step", "algorithmic_bytes_per_launch",
                                                         "dram_over_algorithmic", "all_kernels_dram_bytes_per_step", "gemm_launches_per_step", "source", "command")}
        except Exception:
            pass
        result = {
            "metric": "end-to-end frames/sec (YOLOv8l+UFLDv2+ByteTrack) 1280x720", "value": round(fps, 2), "unit": "frames/s",
            "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": round(ms_dev / K, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": "YOLOv8l 640x640 + UFLDv2-CULane-ResNet34 320x1600 + ByteTrack, 1280x720 synthetic stream per GPU, "
                                   f"batch {B} frames per step (BASELINE configs[3]; configs[4] when n_gpus=8)",
                       "global_batch": world * B, "parallelism": f"dp{world} (one stream per GPU; the detection/track records of EVERY batch are NCCL all-gathered per step, inside the timed region, by the library's own communicator on a private stream)",
                       "weights": "seeded synthetic (He-normal, BN folded), fp16 operands, fp32 accumulate",
                       "l2": f"inputs rotate through a {pool_batches}-batch pool ({pool_batches * B * FRAME_H * FRAME_W * 3 / 1e6:.0f} MB > 126 MB L2)"},
            "e2e": {"value": round(fps_e2e, 2), "unit": "frames/s", "h2d_bytes_per_step": B * FRAME_H * FRAME_W * 3,
                    "d2h_bytes_per_step": int(B * (MAX_DET * (16 + 4 + 4 + 4) + 8) + B * (4 * 81 * 2 * 4 + 16 + 4)),
                    "ms_per_step": round(ms_e2e / K, 4),
                    "note": "adas_b200.pipeline.AdasPipeline.step_pipelined: pinned host batch -> device staging (side stream), both detectors, tracker; results on the host every step"},
            "gpu_launches": int(launches),
            "host_tracker_ms_per_step": round(1e3 * getattr(pipe, "track_seconds", 0.0) / max(1, getattr(pipe, "track_batches", 1)), 3),
            "host_tracker_breakdown_ms_per_step": (lambda st, nb: {"library_total": round(st["total_ms"] / nb, 3), "association_round_trips": round(st["wait_ms"] / nb, 3),
                                                                   "association_launches_per_step": round(st["launches"] / nb, 2)})(
                pipe.tracker._nt.stats(), max(1, getattr(pipe, "track_batches", 1))),
            "tracks_alive": len(pipe.tracker.tracked_stracks),
            "gather": ({"per_step": True, "nccl_ranks": comm.info()[0], "all_gathers": comm.info()[1], "bytes_per_rank_per_step": int(rec.nbytes)} if comm is not None else None),
            "clocks": clocks, "clocks_e2e": clocks_e2e,
            "roofline": {"bound": "tensor", "kernel": "conv_gemm_v3_kernel (tcgen05 implicit-GEMM conv/FC, persistent, warp-specialised, staged TMA-store epilogue)", "achieved": round(achieved, 1), "peak": peak,
                         "unit": "TFLOP/s", "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_detail": traffic_detail,
                         "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst; GEMM launches timed alone, of measured)" if peaks else "fallback 1590 (of fallback)",
                         "launches_per_step": n_y + n_u, "avg_launch_us": round(1e3 * (ms_y + ms_u) / (n_y + n_u), 2),
                         "algorithmic_gflop_per_step": round(gflop_step, 1),
                         "gemm_ms_per_step": round(ms_y + ms_u, 4), "all_plan_kernels_ms_per_step": round(ms_all_y + ms_all_u, 4)},
        }
        # the CPU baseline runs with the pipeline shut down (its worker threads would compete for the host cores and bias the
        # thread-count probe): same conditions as the --impl reference arm
        pipe.close()
        cpu = cpu_baseline_sample(plans, frames=args.cpu_frames) if args.cpu_frames > 0 else None
        if cpu is not None:
            result["cpu_baseline"] = cpu
        if world == 1 and args.other_configs:
            # BASELINE configs[1] / configs[2]: the two conv stacks alone at batch 32 (GEMM launches of one pass, timed like `roofline`)
            other = {}
            for name, key, gf in (("yolov8l_b32 (configs[1])", "yolov8", gf_y), ("ufldv2_res34_b32 (configs[2])", "ufldv2", gf_u)):
                eng = _capi.Engine(plans[key][0], local, max_batch=32)
                ms_g, n_g = eng.time_ops(32, 1 << 1, 3)
                ms_a, _ = eng.time_ops(32, 0xFFFFFFFF, 3)
                eng.close()
                other[name] = {"gemm_tflops": round(gf * 32 / ms_g, 1), "frac_of_peak": round(gf * 32 / ms_g / peak, 4), "gemm_ms": round(ms_g, 3),
                               "all_plan_kernels_ms": round(ms_a, 3), "images_per_s_plan_only": round(32e3 / ms_a, 1), "gemm_launches": n_g}
            result["other_configs"] = other
        print(json.dumps(result), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return result


# ------------------------------------------------------------------------------------------------------------
# the CPU port of the reference path (oracle) -- checker-as-baseline, never the product
# ------------------------------------------------------------------------------------------------------------
class CpuReferencePath:
    def __init__(self, plans):
        import torch
        from oracle import nets, post, track
        self.torch, self.post = torch, post
        self.threads = pick_cpu_threads()
        self.yolo = nets.build("yolov8", plans["yolov8"][1], scale="l")
        self.ufld = nets.build("ufldv2", plans["ufldv2"][1], backbone="34")
        self.trk = track.Tracker()
        self.trk.reset()

    def frame(self, img):
        torch, post = self.torch, self.post
        blob, geom = post.yolo_prepare_input(img, 640, 640)
        with torch.no_grad():
            raw = self.yolo(torch.from_numpy(blob)).numpy()[0]
        det = post.yolo_postprocess(raw, "v8", geom, BOX_SCORE, NMS_IOU)
        x = post.ufld_prepare_input(img, 320, 1600, 0.6)
        with torch.no_grad():
            heads = [o.numpy() for o in self.ufld(torch.from_numpy(x))]
        lanes = post.ufld_decode(heads, img.shape[1], img.shape[0], post.CULANE_ROW_ANCHOR, post.CULANE_COL_ANCHOR)
        b = det["boxes"]
        xyxy = np.stack([b[:, 0], b[:, 1], b[:, 0] + b[:, 2], b[:, 1] + b[:, 3]], 1).astype(int) if len(b) else np.zeros((0, 4), int)
        self.trk.update(xyxy, det["scores"], det["cls"])
        return det, lanes


_CPU_THREADS = None


def pick_cpu_threads() -> int:
    """All the host threads torch can USE: oneDNN convolutions stop scaling (and collapse under oversubscription) well
    before 100+ logical CPUs, so time one conv stack at a few thread counts up to the affinity mask and keep the fastest."""
    global _CPU_THREADS
    import torch
    if _CPU_THREADS is None:
        avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        net = torch.nn.Sequential(torch.nn.Conv2d(64, 128, 3, padding=1), torch.nn.SiLU(), torch.nn.Conv2d(128, 128, 3, padding=1)).eval()
        x = torch.randn(1, 64, 160, 160)
        best, best_t = 1, 1e9
        for n in sorted({c for c in (4, 8, 16, 32, 64, avail) if c <= avail}):
            torch.set_num_threads(n)
            with torch.no_grad():
                net(x)
                t0 = time.perf_counter()
                for _ in range(3):
                    net(x)
                dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = n, dt
        _CPU_THREADS = best
    torch.set_num_threads(_CPU_THREADS)
    return _CPU_THREADS


def cpu_baseline_sample(plans, frames: int = 8):
    path = CpuReferencePath(plans)
    imgs = synth_stream(1000, frames + 1)
    path.frame(imgs[0])                     # warm-up (thread pools, allocator)
    t0 = time.perf_counter()
    for i in range(frames):
        path.frame(imgs[1 + i])
    dt = time.perf_counter() - t0
    return {"value": round(frames / dt, 3), "unit": "frames/s", "cores": path.threads, "kind": "port",
            "sample": f"{frames} consecutive 1280x720 frames, batch 1 (the reference's only mode), oracle port: reference pre/post/tracker "
                      "semantics in numpy + torch-CPU fp32 nets (onnxruntime absent -> torch-CPU substitutes ORT-CPU)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    plans = build_plans()
    path = CpuReferencePath(plans)
    per_step = args.ref_frames
    K, Wm = args.steps, max(args.warmup, 1)
    Wm = min(Wm, 2)                         # at most two warm-up steps: ~1 s of CPU per frame
    imgs = synth_stream(1000, per_step * 4)
    for i in range(Wm):
        for f in range(per_step):
            path.frame(imgs[(i * per_step + f) % len(imgs)])
    t0 = time.perf_counter()
    for i in range(K):
        for f in range(per_step):
            path.frame(imgs[((Wm + i) * per_step + f) % len(imgs)])
    dt = time.perf_counter() - t0
    fps = K * per_step / dt
    sample = (f"each step = {per_step} consecutive 1280x720 frames at batch 1 through the oracle port of the reference path "
              "(torch-CPU fp32 substitutes ONNXRuntime-CPU, which is not installed)")
    print(json.dumps({
        "impl": "reference", "metric": "end-to-end frames/sec (YOLOv8l+UFLDv2+ByteTrack) 1280x720", "value": round(fps, 3), "unit": "frames/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": K, "warmup": Wm, "ms_per_step": round(dt / K * 1e3, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "YOLOv8l 640x640 + UFLDv2-CULane-ResNet34 320x1600 + ByteTrack, 1280x720 synthetic stream (CPU, bounded sample)",
                   "frames_per_step": per_step},
        "cpu_baseline": {"value": round(fps, 3), "unit": "frames/s", "cores": path.threads, "kind": "port", "sample": sample},
        "e2e": {"value": round(fps, 3), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--profile-steps", type=int, default=0, help="profiler target: run N steps between cudaProfilerStart/Stop and exit")
    ap.add_argument("--other-configs", type=int, default=1, help="also time the two conv stacks alone at batch 32 (N=1 only)")
    ap.add_argument("--sets", type=int, default=2, help="engine pairs the pipeline alternates between (batches in flight on the device)")
    ap.add_argument("--depth", type=int, default=3, help="batches queued ahead of the tracker")
    ap.add_argument("--cpu-frames", type=int, default=8, help="frames in the cpu_baseline sample (0 disables)")
    ap.add_argument("--ref-frames", type=int, default=2, help="frames per step of the --impl reference arm")
    ap.add_argument("--watchdog", type=int, default=int(os.environ.get("ADAS_B200_WATCHDOG", "1500")),
                    help="seconds after which a stuck run dumps every thread's stack to stderr and exits non-zero (0 disables)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (detections, lanes, tracks of rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.profile_steps):
        ap.error("--dump-outputs needs the timed steps of --impl b200")
    if not os.environ.get("ADAS_B200_PLAN_CACHE"):
        # the plans are rebuilt from their seeds on every run anyway: write their files to a private temporary directory that is
        # removed at exit, so a run needs no writable home directory and leaves nothing behind
        import atexit
        import shutil
        import tempfile
        tmp = tempfile.mkdtemp(prefix="adas_b200_bench_")
        atexit.register(shutil.rmtree, tmp, True)
        os.environ["ADAS_B200_PLAN_CACHE"] = tmp
    if args.watchdog > 0:
        import faulthandler
        faulthandler.dump_traceback_later(args.watchdog, exit=True, file=sys.stderr)      # a hang must end loudly, with evidence
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
