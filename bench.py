#!/usr/bin/env python
"""bench.py -- throughput of the B200 cuboid-proposal hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3|c2|c4|c5] [--dump-outputs DIR]

A "step" is one pass of the north-star path over one batch of synthetic frames: line segments detected on the device
(line_lbd_detect::detect_filter_lines, LSD flavour -- what object_slam sets, main_obj.cpp:365), then detect_cuboid over
every box of every frame.  N=1 workload: BASELINE config 3 -- 256 synthetic 640x480 frames, ~3 boxes per frame.
N>1 (torchrun, one rank per GPU): every rank processes its own shard of that size (weak scaling), then one NCCL all-gather
of the top-K records.  Prints ONE JSON line on rank 0.

  value         scored (valid) cuboid proposals / s, frames resident in HBM, CUDA-event timed, max over ranks
  e2e           the same through cs_detect_frames_batch with pinned HOST buffers (H2D + kernels + D2H inside)
  roofline      dominant stage: algorithmic bytes / CUDA-event time vs the measured HBM peak
  cpu_baseline  the CPU oracle (a port of the reference's algorithm) on the host cores, same path, bounded sample
  lines_given / online_edlines   the same frames with segments handed in (the detect_cuboid entry point) / with EDLines
--impl reference times the CPU path alone (the reference itself cannot be compiled here: needs Eigen, OpenCV C++ and ROS;
see DESIGN.md): oracle/batch_oracle.cpp, one frame per loop iteration, static schedule over the host cores.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# several batches are kept in flight, three streams each: give the driver enough hardware queues that streams of different batches do not share
# one (the default of 8 makes a long kernel of one batch delay work of another that happens to sit behind it in the same queue)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
# N > 1: every batch ends with an all-gather of < 1 MB of cuboid records on its own stream, two dozen of them in flight.  One NCCL channel
# = one CTA per collective: with the default channel count the waiting all-gather kernels of the batches in flight sat on the SMs the seed
# loops need (measured at N = 2 on one box: 8.29 -> 7.74 ms per step, i.e. 2 x the single-GPU rate)
os.environ.setdefault("NCCL_MAX_NCHANNELS", "1")

WORKLOADS = {
    # name: (frames per GPU, width, height, boxes/frame, kind, poisson, param overrides, description)
    "c2": (1, 640, 480, 5, "indoor", False, {}, "BASELINE config 2: single 640x480 frame, 5 boxes"),
    "c3": (256, 640, 480, 3, "indoor", True, {}, "BASELINE config 3: batch 256 synthetic 640x480 frames, avg 3 boxes/frame"),
    "c4": (128, 1242, 375, 8, "kitti", False, {}, "BASELINE config 4 shard: 128 KITTI-shape 1242x375 frames, 8 boxes/frame per GPU"),
    "c5": (64, 1280, 960, 8, "indoor", False, dict(yaw_step_deg=0.5, top_sample_count_override=30),
           "BASELINE config 5 shard: 64 frames 1280x960, 8 boxes, dense sweep 181 yaw x 30 top-x per GPU"),
}
LINE_LENGTH_THRES = 15.0  # object_slam/src/main_obj.cpp:366

# algorithmic bytes per unit of each stage (DESIGN.md section 4; SURVEY.md section 8d)
STAGE_BYTES = {
    "lsd": lambda s, shp: shp["frame_px"] * s["n_frames"] * 3 + 16 * s["n_lines_in"],  # BGR frame read once + float4 per segment written
    "gray": lambda s, shp: shp["frame_px"] * s["n_frames"] * 4,          # 3 B in + 1 B out per pixel
    "canny": lambda s, shp: s["roi_pixels"] * 2,                           # gray ROI read + edge map written
    "hyst": lambda s, shp: s["roi_pixels"] * 1,                            # edge map, in place
    "dt": lambda s, shp: s["roi_pixels"] * 5,                              # edge map read + f32 dist written
    "lines": lambda s, shp: s["n_lines_in"] * 32 * max(s["n_roi_jobs"], 1) / max(s["n_frames"], 1) + s["n_roi_jobs"] * 56 * 40,
    "sweep": lambda s, shp: s["n_valid"] * 200 + s["n_candidates"] * 1,    # 72 B error row + 128 B corners per scored proposal
    "fuse": lambda s, shp: s["n_valid"] * 16 + s["n_objects"] * 512,
}
STAGE_KERNELS = {"dt": "k_dt_bi<N> (one launch per ROI width class)", "canny": "k_canny_nms", "hyst": "k_canny_hyst", "gray": "k_bgr2gray_flat",
                 "sweep": "k_sweep_warp", "fuse": "k_fuse_warp", "lines": "k_roi_lines",
                 "lsd": "line detector (k_lsd_blur/resize/grad + k_lsd_grow_seq + k_lsd_val_count/nfa x 6 + k_lsd_emit)"}
LIMITERS = {"lsd": "the seed loop (k_lsd_grow_seq, one warp per frame, seeds in raster order) is a dependent chain of L2 / HBM gathers per region pixel: latency-bound, not HBM-bound",
            "canny": "integer ALU pipe (ncu, profiles/): not an HBM-bound kernel",
            "dt": "dependency chain of H row steps per ROI (latency), DRAM traffic below the algorithmic bytes"}


def path_alg_bytes(stats, shp, topk):
    """SURVEY.md section 8(d): W*H*3 + 16*M + sum 6*ROI_px + 200*P_valid + 512*N*topk, per batch."""
    return (shp["frame_px"] * stats["n_frames"] * 3 + 16 * stats["n_lines_in"] + 6 * stats["roi_pixels"] + 200 * stats["n_valid"] +
            512 * stats["n_objects"] * topk)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def physical_cores():
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    return os.cpu_count() or 1


def cpu_quota():
    """CPUs' worth of time the container may use (cgroup cpu.max / cfs quota), or None when unlimited."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            return float(q) / float(per)
    except (OSError, ValueError):
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return q / per
    except (OSError, ValueError):
        pass
    return None


def cpu_thread_choices():
    """Thread counts worth trying for the CPU arm: the logical CPUs, unless a cgroup quota caps the process below that (more runnable threads
    than the quota allows only get throttled): then the quota and twice the quota."""
    logical = os.cpu_count() or 1
    q = cpu_quota()
    if q is None or q >= logical:
        return sorted({logical, physical_cores()})
    base = max(1, int(round(q)))
    return sorted({min(logical, base), min(logical, 2 * base)})


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.rows = []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = max((int(r[1]) for r in self.rows if r[1].isdigit()), default=None)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(self.rows)}


def time_lbd_subprocess():
    """The descriptor / matcher half of line_lbd_detect (SURVEY.md section 8 f4), timed by tools/time_lbd.py in a process of its own after
    the timed region (whatever happens there cannot touch the numbers above); its JSON object, or why there is none."""
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "time_lbd.py")], capture_output=True, text=True, timeout=240)
        if r.returncode != 0:
            return {"error": (r.stderr or r.stdout).strip().splitlines()[-1][:300] if (r.stderr or r.stdout).strip() else "exit %d" % r.returncode}
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:  # noqa: BLE001 -- an extra key must never cost the bench line
        return {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}


def lbd_cpu_one_core(wl, n=4):
    """The descriptor half on one host core, for the `lbd` key: the oracle port of detect_descrip_lines (LSD flavour) and of
    match_line_descrip on n frames of the workload (cpu_baseline leg: the one place bench.py runs oracle code)."""
    try:
        from oracle import pyoracle as O
        imgs = wl["imgs"][:n]
        t0 = time.perf_counter()
        kls = [O.lbd_detect_keylines(im, True, 15.0) for im in imgs]
        t1 = time.perf_counter()
        descs = [O.lbd_compute(im, k) for im, k in zip(imgs, kls)]
        t2 = time.perf_counter()
        pairs = 0
        for q, t in zip(descs[:-1], descs[1:]):
            O.lbd_match(q, t, 40.0)
            pairs += len(q) * len(t)
        t3 = time.perf_counter()
        lines = sum(len(k) for k in kls)
        return {"kind": "port", "cores": 1, "frames": len(imgs), "lines": lines, "describe_lines_per_s": lines / max(t2 - t1, 1e-9),
                "detect_descrip_frames_per_s": len(imgs) / max(t2 - t0, 1e-9), "match_code_pairs_per_s": pairs / max(t3 - t2, 1e-9)}
    except Exception as e:  # noqa: BLE001
        return {"error": "%s: %s" % (type(e).__name__, str(e)[:200])}


def make_workload(name, rank, seed_base=20260922, frames=None):
    from cube_slam_b200 import synthetic as S
    F, w, h, nb, kind, poisson, over, desc = WORKLOADS[name]
    if frames:
        F = frames
    imgs, Ts, boxes, lines, K = S.make_batch(seed_base + 1000 * rank + sum(map(ord, name)), F, w, h, nb, kind=kind, poisson=poisson,
                                             distinct=min(F, 32))
    return dict(imgs=imgs, Ts=Ts, boxes=boxes, lines=lines, K=K, over=over, desc=desc, w=w, h=h, F=F, name=name)


def workload_shape(wl, stats=None):
    allb = np.concatenate([np.asarray(b).reshape(-1, 5) for b in wl["boxes"]])
    d = {"mean_box_w": float(allb[:, 2].mean()), "mean_box_h": float(allb[:, 3].mean()), "boxes_per_frame": len(allb) / wl["F"]}
    if stats:
        d["segments_per_frame_M"] = stats["n_lines_in"] / max(stats["n_frames"], 1)
        d["mean_roi_px"] = stats["roi_pixels"] / max(stats["n_roi_jobs"], 1)
    return d


# ------------------------------------------------------------------------------------------- CPU arm
def cpu_run(wl, n_frames, n_threads, line_mode=1):
    """The reference's per-frame path on the host (oracle port; oracle/batch_oracle.cpp): detect_filter_lines (LSD) then
    detect_cuboid, one frame per loop iteration, static schedule over n_threads.  Returns (seconds, valid, candidates, segments)."""
    from oracle import pyoracle as O
    p = O.default_params(**wl["over"])
    O.lib()
    ids = slice(0, n_frames)
    t0 = time.perf_counter()
    r = O.detect_frames_batch(wl["imgs"][ids], wl["K"], wl["Ts"][ids], wl["boxes"][ids], wl["lines"][ids] if line_mode == 0 else None, p,
                              line_mode=line_mode, line_length_thres=LINE_LENGTH_THRES, n_threads=n_threads)
    dt = time.perf_counter() - t0
    return dt, int(r["n_valid"].sum()), int(r["n_cand"].sum()), int(r["n_lines"].sum())


def lsd_reference_vs_port(wl, n=4):
    """One core, the first n frames: the reference's own lsd.cpp (oracle/_ref/liblsd_ref.so, compiled from the reference where that
    exists) beside the oracle's restatement of it, which the batch driver of the CPU arm runs.  Same segments (tests); ms per frame."""
    from oracle import pyoracle as O
    if not O.ref_lsd_available():
        return None
    frames = [np.ascontiguousarray(O.bgr2gray(wl["imgs"][i])) for i in range(min(n, wl["F"]))]
    O.ref_lsd_detect(frames[0])
    O.lsd_detect(frames[0], LINE_LENGTH_THRES)
    t0 = time.perf_counter()
    for g in frames:
        O.ref_lsd_detect(g)
    t1 = time.perf_counter()
    for g in frames:
        O.lsd_detect(g, LINE_LENGTH_THRES)
    t2 = time.perf_counter()
    return {"reference_lsd_cpp_ms_per_frame": 1e3 * (t1 - t0) / len(frames), "port_ms_per_frame": 1e3 * (t2 - t1) / len(frames), "frames": len(frames),
            "note": "createLineSegmentDetector(LSD_REFINE_ADV)->detect on the gray frame, one core; the reference's lsd.cpp compiled against "
                    "oracle/ref/minicv.hpp vs the oracle port the CPU arm runs"}


def cpu_line_mode():
    """3 = stage (i) by the reference's own detect_filter_lines (oracle/_ref/liblinelbd_ref.so, compiled from the reference's sources where
    that checkout existed), stage (ii) by the oracle port; 1 = the oracle port for both (the reference library is not there)."""
    from oracle import pyoracle as O
    return 3 if O.lib().orc_reference_lines_available() else 1


CPU_KIND = {3: "reference", 1: "port"}
CPU_KIND_NOTE = {
    3: "stage (i), line_lbd_detect::detect_filter_lines: the reference's OWN code (lsd.cpp, LSDDetector.cpp, binary_descriptor.cpp, line_lbd_allclass.cpp "
       "compiled from its sources against oracle/ref/minicv.hpp, oracle/_ref/liblinelbd_ref.so); stage (ii), detect_cuboid: the oracle port "
       "(detect_3d_cuboid needs Eigen, which this image does not have)",
    1: "CPU oracle port of the reference algorithm for both stages (oracle/_ref was not built: no reference checkout at build time)"}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    from oracle import pyoracle as O
    wl = make_workload(args.workload, 0)
    phys = physical_cores()
    mode = cpu_line_mode()
    dt1, _, _, _ = cpu_run(wl, min(wl["F"], 2), 1, mode)
    per_frame = dt1 / min(wl["F"], 2)
    n = int(max(1, min(wl["F"], 4.0 * phys / max(per_frame, 1e-4))))  # about 4 s of wall clock per step at most
    # all the host threads the process can use: the best of the candidate thread counts (cgroup quota aware), measured
    best = None
    for th in cpu_thread_choices():
        cpu_run(wl, n, th, mode)  # the same frames on the same threads: warms every thread's malloc arena
        dt = cpu_run(wl, n, th, mode)[0]
        if best is None or dt < best[0]:
            best = (dt, th)
    threads = best[1]
    for _ in range(max(0, min(args.warmup, 2) - 1)):
        cpu_run(wl, n, threads, mode)
    port_dt = cpu_run(wl, n, threads, 1)[0] if mode != 1 else None  # the all-port arm on the same frames and threads, for the record
    tot_t = tot_v = tot_c = tot_l = 0.0
    for _ in range(args.steps):
        dt, v, c, l = cpu_run(wl, n, threads, mode)
        tot_t += dt
        tot_v += v
        tot_c += c
        tot_l += l
    val = tot_v / tot_t
    fps = n * args.steps / tot_t
    line = {
        "impl": "reference", "metric": "scored cuboid proposals/s", "value": val, "unit": "proposals/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "frames_per_s": fps, "candidates_per_s": tot_c / tot_t,
        "config": {"workload": wl["desc"], "lines": "detected per frame by the LSD flavour of line_lbd (the north-star path)",
                   "sample_frames_per_step": n, "segments_per_frame_M": tot_l / (n * args.steps),
                   "note": CPU_KIND_NOTE[mode] + "; oracle/batch_oracle.cpp, one frame per loop iteration, static schedule, openmp=%d" % O.lib().orc_has_openmp()},
        "cpu_baseline": {"value": val, "unit": "proposals/s", "cores": threads, "physical_cores": phys, "logical_cpus": os.cpu_count(),
                         "cgroup_cpu_quota": cpu_quota(), "cpu": cpu_model(), "kind": CPU_KIND[mode], "kind_detail": CPU_KIND_NOTE[mode],
                         "all_port_frames_per_s": (n / port_dt) if port_dt else None, "one_core_frames_per_s": 1.0 / per_frame,
                         "scaling_vs_one_core": fps * per_frame, "lsd_stage_one_core": lsd_reference_vs_port(wl),
                         "sample": "%d of %d frames per step, line detection + detect_cuboid per frame, %d threads" % (n, wl["F"], threads)},
        "e2e": {"value": val, "unit": "proposals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------- GPU arm
class Mode(object):
    """One way of feeding the same frames through the path on a set of contexts driven round-robin."""

    def __init__(self, name, ctxs, streams, wl, params, line_params=None):
        self.name, self.ctxs, self.streams, self.wl, self.params, self.lp = name, ctxs, streams, wl, params, line_params

    def upload(self, which=None):
        wl = self.wl
        for cx in (self.ctxs if which is None else which):
            if self.lp is None:
                cx.upload(wl["imgs"], wl["Ts"], wl["boxes"], wl["lines"], self.params)
            else:
                cx.upload_online(wl["imgs"], wl["Ts"], wl["boxes"], self.lp, self.params)


def dump_outputs(out_dir, cx):
    """--dump-outputs: what a caller of the timed path receives for the batch of its last step (cs_batch_fetch): the top-K cuboid records
    of every object, one float64 array per record field (objects x K [x field shape]; slots past an object's count are zero), and the
    count of each object."""
    recs, counts = cx.fetch()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "counts.npy"), counts.astype(np.float64))
    for name in recs.dtype.names:
        if name != "pad_":
            np.save(os.path.join(out_dir, "cuboid_%s.npy" % name), recs[name].astype(np.float64))


def make_line_params(cs, cx, use_lsd=True):
    det = cs.line_lbd_detect(context=cx)
    det.use_LSD = use_lsd
    det.line_length_thres = LINE_LENGTH_THRES
    return det.params()


def nccl_library_path():
    for d in sys.path:
        cand = os.path.join(d, "nvidia", "nccl", "lib", "libnccl.so.2")
        if os.path.exists(cand):
            return cand
    return ""


def init_comm(cx, rank, world, dist, torch, _lib):
    """The library's own NCCL communicator for this context: unique id from rank 0, broadcast over torch.distributed."""
    path = nccl_library_path().encode()
    uid = np.zeros(128, np.uint8)
    if rank == 0:
        cx.check(cx.L.cs_comm_unique_id(cx.h, path, _lib.ptr(uid, C.c_uint8)))
    t = torch.from_numpy(uid).cuda()
    dist.broadcast(t, 0)
    uid = t.cpu().numpy()
    cx.check(cx.L.cs_comm_init(cx.h, path, _lib.ptr(uid, C.c_uint8), world, rank))


def measure_config(name, args, rank, world, local_rank, dist, cs, _lib, torch):
    """One of the other BASELINE configurations at this rank count: every rank holds its shard (WORKLOADS[name] frames per GPU), twelve batches in
    flight (with the all-gather of N > 1 coupling the ranks batch by batch, six were too few to hide the wait for the slower rank), online LSD lines, the top-K all-gather inside every step when N > 1.  Returns the dict that goes under the config's key."""
    wl = make_workload(name, rank)
    F, w, h = wl["F"], wl["w"], wl["h"]
    params = cs.default_params(**wl["over"])
    topk = int(params.max_cuboid_num)
    ctxs = []
    for _ in range(12):
        cx = cs.Context(local_rank, w, h, F, 16, 8192)
        cx.set_calibration(wl["K"])
        ctxs.append(cx)
    dev = torch.device("cuda", local_rank)
    streams = [torch.cuda.ExternalStream(cx.stream(), device=dev) for cx in ctxs]
    recs_per_rank = 0
    if world > 1:
        for cx in ctxs:
            init_comm(cx, rank, world, dist, torch, _lib)
        n_obj = torch.tensor([sum(len(b) for b in wl["boxes"])], device="cuda")
        dist.all_reduce(n_obj, op=dist.ReduceOp.MAX)
        recs_per_rank = int(n_obj.item()) * topk
    lp = make_line_params(cs, ctxs[0])
    for cx in ctxs:
        cx.upload_online(wl["imgs"], wl["Ts"], wl["boxes"], lp, params)
    gathered = C.c_void_p()

    def step_i(i):
        cx = ctxs[i % len(ctxs)]
        cx.run_async()
        if world > 1:
            cx.check(cx.L.cs_allgather_topk(cx.h, recs_per_rank, C.byref(gathered)))

    steps = 2 * len(ctxs)
    for i in range(2 * len(ctxs)):
        step_i(i)
    torch.cuda.synchronize()
    st = ctxs[0].stats()
    ev0 = torch.cuda.Event(enable_timing=True)
    ev_end = [torch.cuda.Event(enable_timing=True) for _ in ctxs]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0.record(streams[0])
    for s_ in streams[1:]:
        s_.wait_event(ev0)
    for i in range(steps):
        step_i(i)
    if world > 1:  # the collectives run on the contexts' gather streams: the end events go behind the last one of each context
        for cx in ctxs:
            cx.check(cx.L.cs_allgather_wait(cx.h))
    for e, s_ in zip(ev_end, streams):
        e.record(s_)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = max(ev0.elapsed_time(e) for e in ev_end) / steps
    t = torch.tensor([ms, float(st["n_valid"]), float(st["n_candidates"]), float(st["n_frames"]), float(st["n_objects"])], device="cuda", dtype=torch.float64)
    allt = [t.clone()]
    if world > 1:
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
    for cx in ctxs:
        cx.close()
    ms_max = max(float(x[0].item()) for x in allt)
    valid = sum(float(x[1].item()) for x in allt)
    frames = sum(float(x[3].item()) for x in allt)
    return {"workload": wl["desc"], "ms_per_step": ms_max, "value": valid / (ms_max * 1e-3), "unit": "proposals/s", "frames_per_s": frames / (ms_max * 1e-3),
            "candidates_per_s": sum(float(x[2].item()) for x in allt) / (ms_max * 1e-3), "steps": steps, "batches_in_flight": len(ctxs),
            "frames_per_gpu": F, "boxes_total": sum(float(x[4].item()) for x in allt), "segments_per_frame_M": st["n_lines_in"] / max(st["n_frames"], 1),
            "per_rank_ms_per_step": [float(x[0].item()) for x in allt]}


def run_ours(args, rank, world, local_rank):
    import torch
    import cube_slam_b200 as cs
    from cube_slam_b200 import _lib
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    wl = make_workload(args.workload, rank)
    F, w, h = wl["F"], wl["w"], wl["h"]
    params = cs.default_params(**wl["over"])
    topk = int(params.max_cuboid_num)
    n_ctx = max(args.inflight, 1)
    ctxs = []
    for _ in range(n_ctx):
        cx = cs.Context(local_rank, w, h, F, 16, 8192)
        cx.set_calibration(wl["K"])
        ctxs.append(cx)
    ctx = ctxs[0]
    streams = [torch.cuda.ExternalStream(cx.stream(), device=dev) for cx in ctxs]
    dbg_flags = (16 if args.no_prio else 0) | (32 if args.raster_dt else 0) | (128 if args.seq_lines else 0)

    def line_params(use_lsd):
        det = cs.line_lbd_detect(context=ctx)
        det.use_LSD = use_lsd
        det.line_length_thres = LINE_LENGTH_THRES
        return det.params()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    gathered = C.c_void_p()
    recs_per_rank = 0
    if world > 1:
        for cx in ctxs:
            init_comm(cx, rank, world, dist, torch, _lib)
        n_obj = torch.tensor([sum(len(b) for b in wl["boxes"])], device="cuda")
        dist.all_reduce(n_obj, op=dist.ReduceOp.MAX)
        recs_per_rank = int(n_obj.item()) * topk

    def timed(mode, steps, warm, with_gather):
        """warm-up, then `steps` steps round-robin over the contexts; device time (ms, this rank) and the batch statistics."""
        mode.upload()
        for cx in ctxs:
            cx.set_profiling(dbg_flags)

        def step_i(i):
            cx = ctxs[i % len(ctxs)]
            cx.run_async()
            if with_gather:
                cx.check(cx.L.cs_allgather_topk(cx.h, recs_per_rank, C.byref(gathered)))

        def join_gathers():
            # the collectives run on the contexts' gather streams: order each context stream behind its last one before the end events
            if with_gather:
                for cx in ctxs:
                    cx.check(cx.L.cs_allgather_wait(cx.h))

        for i in range(max(warm, 3) * len(ctxs)):
            step_i(i)
        torch.cuda.synchronize()
        st = ctx.stats()
        ev0 = torch.cuda.Event(enable_timing=True)
        ev_end = [torch.cuda.Event(enable_timing=True) for _ in ctxs]
        barrier()
        ev0.record(streams[0])
        for s_ in streams[1:]:
            s_.wait_event(ev0)
        for i in range(steps):
            step_i(i)
        join_gathers()
        for e, s_ in zip(ev_end, streams):
            e.record(s_)
        barrier()
        ms = max(ev0.elapsed_time(e) for e in ev_end)
        # one more step alone, profiled: latency of a batch and its stage times
        ctx.set_profiling(1 | dbg_flags)
        ctx.run()
        stage = ctx.stage_ms()
        ctx.set_profiling(dbg_flags)
        if with_gather:  # the all-gather alone, CUDA events on the context's stream
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            g0.record(streams[0])
            ctx.check(ctx.L.cs_allgather_topk(ctx.h, recs_per_rank, C.byref(gathered)))
            ctx.check(ctx.L.cs_allgather_wait(ctx.h))
            g1.record(streams[0])
            torch.cuda.synchronize()
            stage["allgather"] = g0.elapsed_time(g1)
        return ms, st, stage

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    main_mode = Mode("online_lsd", ctxs, streams, wl, params, line_params(True))
    ms_total, stats, stage_acc = timed(main_mode, args.steps, args.warmup, world > 1)
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctxs[(args.steps - 1) % len(ctxs)])
    my_ms = ms_total
    ms_t = torch.tensor([ms_total], device="cuda", dtype=torch.float64)
    cnt = torch.tensor([stats["n_valid"], stats["n_candidates"], stats["n_frames"], stats["n_objects"]], device="cuda", dtype=torch.float64)
    per_rank = None
    if world > 1:
        allms = [torch.zeros_like(ms_t) for _ in range(world)]
        dist.all_gather(allms, ms_t)
        allcnt = [torch.zeros_like(cnt) for _ in range(world)]
        dist.all_gather(allcnt, cnt)
        per_rank = {"ms_per_step": [float(x.item()) / args.steps for x in allms], "boxes": [float(x[3].item()) for x in allcnt],
                    "valid": [float(x[0].item()) for x in allcnt], "allgather_ms_rank0": stage_acc.get("allgather"),
                    "allgather_bytes_per_rank": recs_per_rank * cs.CUBOID_DTYPE.itemsize}
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    ms_total = float(ms_t.item())
    n_valid_all, n_cand_all, n_frames_all, n_obj_all = [float(x) for x in cnt.tolist()]
    ms_per_step = ms_total / args.steps
    value = n_valid_all / (ms_per_step * 1e-3)

    # ---- the same frames, other entry points (N = 1 only): segments handed in; EDLines instead of LSD
    extra = {}
    if world == 1 and not args.no_extra:
        sub_steps = max(20, min(args.steps, 200))
        for name, mode in (("lines_given", Mode("lines_given", ctxs, streams, wl, params, None)),
                           ("online_edlines", Mode("online_edlines", ctxs, streams, wl, params, line_params(False)))):
            ms_x, st_x, stage_x = timed(mode, sub_steps, 3, False)
            extra[name] = {"ms_per_step": ms_x / sub_steps, "value": st_x["n_valid"] / (ms_x / sub_steps * 1e-3), "unit": "proposals/s",
                           "frames_per_s": F / (ms_x / sub_steps * 1e-3), "n_valid": st_x["n_valid"], "segments_per_frame_M": st_x["n_lines_in"] / F,
                           "one_batch_alone_ms": stage_x.get("total"), "stage_ms": stage_x}
        extra["lines_given"]["workload"] = "segments given as input (the detect_cuboid entry point; how orb_object_slam feeds it, Tracking.cc:1583-1590)"
        extra["online_edlines"]["workload"] = "lines from the EDLines flavour (use_LSD = false, the class default), length > 15"
        main_mode.upload()

    # ---- end to end through the host-buffer ABI call ("e2e"): cs_detect_frames_batch, pinned host frames
    pinned = torch.from_numpy(wl["imgs"]).pin_memory()
    imgs_pinned = pinned.numpy()
    n_obj_loc = max(int(stats["n_objects"]), 1)
    # host threads, one context each, call the synchronous ABI entry point: the copies of one batch overlap the kernels of the others
    # (single GPU only: two threads issuing NCCL calls on two communicators in an unordered way could deadlock across ranks)
    e2e_ctxs = ctxs if (len(ctxs) >= 2 and world == 1) else ctxs[:1]
    e2e_out = [(np.zeros((n_obj_loc, topk), cs.CUBOID_DTYPE), np.zeros(n_obj_loc, np.int32)) for _ in e2e_ctxs]
    lp_main = main_mode.lp

    def step_e2e(k=0):
        cx = e2e_ctxs[k]
        cx.detect_frames_host(imgs_pinned, wl["Ts"], wl["boxes"], lp_main, params, e2e_out[k][0], e2e_out[k][1])
        if world > 1:
            cx.check(cx.L.cs_allgather_topk(cx.h, recs_per_rank, C.byref(C.c_void_p())))

    e2e_mode = "host threads, one context each, cs_detect_frames_batch (synchronous)"
    if world == 1:
        for k in range(len(e2e_ctxs)):
            for _ in range(2):
                step_e2e(k)
        barrier()
        # enough rounds per thread that filling and draining the pipeline (a batch alone takes ~55 ms) does not dominate
        e2e_steps = max(args.steps, 8 * len(e2e_ctxs))
        e2e_steps -= e2e_steps % len(e2e_ctxs)

        def e2e_worker(k):
            torch.cuda.set_device(local_rank)
            for _ in range(e2e_steps // len(e2e_ctxs)):
                step_e2e(k)

        t0 = time.perf_counter()
        workers = [threading.Thread(target=e2e_worker, args=(k,)) for k in range(len(e2e_ctxs))]
        for t in workers:
            t.start()
        for t in workers:
            t.join()
        barrier()
        e2e_ms = (time.perf_counter() - t0) * 1e3  # host-synchronous calls: the wall clock around all of them is the honest bound
        e2e_sync = {"ms_per_step": e2e_ms / e2e_steps, "frames_per_s": n_frames_all / (e2e_ms / e2e_steps * 1e-3), "steps": e2e_steps,
                    "host_threads": len(e2e_ctxs), "mode": e2e_mode}
    else:
        e2e_sync = None
    if True:
        # The pipelined form of the same ABI (every N): one host thread keeps the batches in flight with the split calls --
        # cs_batch_upload_online (pinned host frames -> device, tables), cs_batch_run_async, cs_allgather_topk when N > 1, cs_batch_fetch
        # (records -> host) -- as a rolling pipeline: step s is issued on context s mod K, then the oldest outstanding step is fetched.  Every
        # rank issues its collectives in the same order, and no host thread sleeps in a synchronous call while its context could be copying.
        e2e_ctxs = ctxs
        K_ = len(e2e_ctxs)
        e2e_mode = "one host thread, %d contexts as a rolling pipeline: cs_batch_upload_online + cs_batch_run_async%s + cs_batch_fetch" % (
            K_, " + cs_allgather_topk" if world > 1 else "")

        def e2e_issue(cx):
            cx.upload_online(imgs_pinned, wl["Ts"], wl["boxes"], lp_main, params)
            cx.run_async()
            if world > 1:
                cx.check(cx.L.cs_allgather_topk(cx.h, recs_per_rank, C.byref(C.c_void_p())))

        def e2e_run(n_steps):
            issued = fetched = 0
            while fetched < n_steps:
                while issued < n_steps and issued - fetched < K_:
                    e2e_issue(e2e_ctxs[issued % K_])
                    issued += 1
                if world > 1:  # a step is complete when its all-gather is: order the fetch behind it
                    e2e_ctxs[fetched % K_].check(e2e_ctxs[fetched % K_].L.cs_allgather_wait(e2e_ctxs[fetched % K_].h))
                e2e_ctxs[fetched % K_].fetch()
                fetched += 1

        e2e_run(K_)
        barrier()
        e2e_steps = max(args.steps, 8 * K_)
        t0 = time.perf_counter()
        e2e_run(e2e_steps)
        barrier()
        e2e_ms = (time.perf_counter() - t0) * 1e3
    e2e_t = torch.tensor([e2e_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_ms_step = float(e2e_t.item()) / e2e_steps
    h2d = wl["imgs"].nbytes + wl["Ts"].nbytes + sum(np.asarray(b).nbytes for b in wl["boxes"])
    d2h = e2e_out[0][0].nbytes + e2e_out[0][1].nbytes

    # ---- the other north-star configurations (BASELINE configs 4 and 5), a short run each, same protocol (online LSD, all-gather when N > 1)
    other = {}
    if not args.no_configs and args.workload == "c3":
        for cx in ctxs:
            cx.close()
        ctxs = []
        for name in ("c4", "c5"):
            other[name] = measure_config(name, args, rank, world, local_rank, dist, cs, _lib, torch)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant stage
    hbm_peak, peak_src = measured_peaks()
    shp = {"frame_px": w * h}
    kernel_ms = {k: v for k, v in stage_acc.items() if k not in ("total", "allgather")}
    dom = max(kernel_ms, key=kernel_ms.get)
    dom_bytes = float(STAGE_BYTES[dom](stats, shp))
    achieved = dom_bytes / (kernel_ms[dom] * 1e-3) / 1e9 if kernel_ms[dom] > 0 else 0.0
    path_bytes = float(path_alg_bytes(stats, shp, topk))
    traffic = None  # DRAM bytes of the stage's kernels per launch, from the committed ncu capture of this workload (profiles/)
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        traffic = tj.get(args.workload, {}).get(dom)
    except (OSError, ValueError):
        pass
    roofline = {"bound": "hbm", "kernel": "%s: %s" % (dom, STAGE_KERNELS.get(dom, dom)), "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": traffic, "limiter": LIMITERS.get(dom), "peak_source": peak_src, "alg_bytes_per_launch": dom_bytes,
                "path": {"alg_bytes_per_step": path_bytes, "achieved": path_bytes / (ms_per_step * 1e-3) / 1e9,
                         "frac": path_bytes / (ms_per_step * 1e-3) / 1e9 / hbm_peak},
                "stage_ms": stage_acc,
                "stage_gbs": {k: float(STAGE_BYTES[k](stats, shp)) / (v * 1e-3) / 1e9 for k, v in kernel_ms.items() if v > 0}}

    # ---- CPU baseline (rank 0, N=1 only), bounded sample of the same workload, same path (line detection + detect_cuboid)
    cpu = None
    if world == 1 and not args.no_cpu:
        from oracle import pyoracle as O
        phys = physical_cores()
        mode = cpu_line_mode()
        dt1, v1, _, _ = cpu_run(wl, min(F, 4), 1, mode)
        per_frame = dt1 / min(F, 4)
        n = int(max(1, min(F, 10.0 * phys / max(per_frame, 1e-4))))
        tried = {}
        for th in cpu_thread_choices():
            cpu_run(wl, n, th, mode)  # warm-up on every thread
            tried[th] = min((cpu_run(wl, n, th, mode) for _ in range(2)), key=lambda r: r[0])
        threads = min(tried, key=lambda t: tried[t][0])
        dt, v, c, l = tried[threads]
        port_dt = cpu_run(wl, n, threads, 1)[0] if mode != 1 else None
        cpu = {"value": v / dt, "unit": "proposals/s", "cores": threads, "physical_cores": phys, "logical_cpus": os.cpu_count(), "cgroup_cpu_quota": cpu_quota(),
               "cpu": cpu_model(), "kind": CPU_KIND[mode], "kind_detail": CPU_KIND_NOTE[mode], "all_port_frames_per_s": (n / port_dt) if port_dt else None,
               "frames_per_s": n / dt, "one_core_value": v1 / dt1, "one_core_frames_per_s": 1.0 / per_frame,
               "scaling_vs_one_core": (v / dt) / (v1 / dt1), "frames_per_s_by_threads": {str(t): n / r[0] for t, r in tried.items()},
               "openmp": int(O.lib().orc_has_openmp()), "lsd_stage_one_core": lsd_reference_vs_port(wl),
               "sample": "%d of %d frames of this workload, LSD line detection + detect_cuboid per frame, static schedule, %d threads (the best of %s; "
                         "the box caps the process at %s CPUs' worth of time)" % (n, F, threads, sorted(tried), cpu_quota())}

    line = {
        "metric": "scored cuboid proposals/s", "value": value, "unit": "proposals/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "frames_per_s": n_frames_all / (ms_per_step * 1e-3), "candidates_per_s": n_cand_all / (ms_per_step * 1e-3),
        "config": dict({"workload": wl["desc"], "frames_per_gpu": F, "boxes_total": n_obj_all, "valid_fraction": n_valid_all / max(n_cand_all, 1),
                        "lines": "detected on the device from the resident frames: line_lbd_detect::detect_filter_lines, LSD flavour, length > 15 (stage (i) of the north star)",
                        "l2": "inputs larger than L2 (%.0f MB of frames per GPU)" % (wl["imgs"].nbytes / 1e6),
                        "parallelism": "frames sharded x%d, one NCCL all-gather of top-K" % world if world > 1 else "single GPU",
                        "batches_in_flight": n_ctx, "one_batch_alone_ms": stage_acc.get("total")}, **workload_shape(wl, stats)),
        "e2e": {"value": n_valid_all / (e2e_ms_step * 1e-3), "unit": "proposals/s", "frames_per_s": n_frames_all / (e2e_ms_step * 1e-3),
                "ms_per_step": e2e_ms_step, "steps": e2e_steps, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "host_threads": 1, "batches_in_flight": len(e2e_ctxs), "mode": e2e_mode, "sync_calls": e2e_sync,
                "timer": "wall clock around all calls"},
        "gpu_launches": int(stats["n_kernel_launches"]) * args.steps,
        "roofline": roofline, "cpu_baseline": cpu, "clocks": sampler.summary(),
    }
    line.update(extra)
    line.update(other)
    if per_rank:
        line["per_rank"] = per_rank
    if world == 1 and not args.no_extra:
        line["lbd"] = time_lbd_subprocess()
        if not args.no_cpu:
            line["lbd"]["cpu_one_core"] = lbd_cpu_one_core(wl)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the lines-given / EDLines variants of the same frames")
    ap.add_argument("--no-configs", action="store_true", help="skip the short runs of BASELINE configs 4 and 5 (keys c4, c5)")
    ap.add_argument("--no-prio", action="store_true", help="A/B: keep each batch's whole chain on one stream (no high-priority tail)")
    ap.add_argument("--raster-dt", action="store_true", help="A/B: two-pass raster-scan distance transform kernel instead of the cone form")
    ap.add_argument("--seq-lines", action="store_true", help="A/B: the line detectors' sequential kernels (one warp per frame) instead of ordered speculation")
    ap.add_argument("--inflight", type=int, default=24, help="batches in flight on one GPU (contexts driven round-robin)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the cuboid records of the last step's batch (rank 0) "
                    "to DIR/<name>.npy, float64, for comparing two builds on the same seeded inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    if args.steps is None:
        args.steps = 300 if args.impl == "ours" else 3
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # convenience: python bench.py --gpus N re-launches itself under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
               "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
