#!/usr/bin/env python3
"""bench.py -- Mkeypoints/s of the ORB front-end hot path (extract + match) on B200.

Workload (BASELINE.json configs[1]): a stream of synthetic 1920x1080 u8 frames, ORBextractor(2000, 1.2, 8,
FAST_SCORE, 20), frame-to-frame ORBmatcher(0.9, true).SearchByProjection(Current, Last, 15).
One "step" = `--frames` DISTINCT consecutive frames of the stream per GPU (default 256 = 531 MB of pixels, 4.2x the
126 MB L2), processed as `--frames / --batch` batches of `--batch` frames and `--repeat` passes over them (default 4:
a step is then 1024 frame extractions + matches, ~51 ms of GPU work, 20 steps time >= 1 s): extract every frame, match every frame against
its predecessor.  Mkeypoints/s = keypoints extracted-and-matched / time.

  value : inputs already resident in HBM when the timed region starts (device API of liborbfe.so),
          results read back + matched.
  e2e   : the reference-facing C-ABI call with HOST buffers (orbfe_extract_batch + the matcher), H2D of the
          step's frames from pinned memory and D2H of keypoints/descriptors inside the timed region.

`--impl reference` times the CPU oracle port of the reference path (oracle/) on the host cores.
`--dump-outputs DIR` writes what the value path returned in the last timed step, for a fixed sample of the step's frames, as
DIR/<name>.npy (float32); the inputs are seeded, so two builds run with the same arguments can be compared output for output.
PyTorch is used only for plumbing: device buffers, pinned host memory, torch.distributed.
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

W, H, NFEAT, NLEVELS, SCALE, FAST_TH = 1920, 1080, 2000, 8, 1.2, 20
FX = FY = 1000.0
CX, CY = W / 2.0, H / 2.0
DEPTH = 5.0
MATCH_TH = 15.0  # Tracking.cc:565
DUMP_FRAMES = 32  # frames of the last step written by --dump-outputs: 32 x 2000 keypoints x 40 floats = 10 MB
METRIC = "Mkeypoints/s extract+match"


def level_sizes():
    # float32 emulation of ORBextractor.cc:461-471,785-786
    inv = np.float32(1.0) / np.float64(np.float32(SCALE))
    inv = np.float32(inv)
    s = np.float32(1.0)
    out = []
    for l in range(NLEVELS):
        out.append((int(np.rint(np.float32(W) * s)), int(np.rint(np.float32(H) * s))))
        s = np.float32(s * inv)
    return out


def algorithmic_bytes():
    """SURVEY.md 8(d): per-frame algorithmic bytes of extract (reads, writes, gathers, outputs)."""
    ls = level_sizes()
    P = sum(w * h for w, h in ls)
    reads = sum(w * h for w, h in ls[:-1]) + 2 * P
    writes = (P - W * H) + P
    gathers = NFEAT * (749 + 512)
    outputs = NFEAT * 60
    return {"P": P, "total": reads + writes + gathers + outputs, "fast_read": P, "blur": 2 * P,
            "resize": sum(w * h for w, h in ls[:-1]) + (P - W * H)}


def make_stream(nframes, seed, per_base=32):
    """`nframes` consecutive DISTINCT frames: a new base texture every `per_base` frames (a scene cut), each followed by
    small random translations of its predecessor plus fresh sensor noise (so no two frames share pixel values)."""
    from concurrent.futures import ThreadPoolExecutor
    from orb_slam_b200.synth import textured_frame, shifted_frame
    frames = np.empty((nframes, H, W), np.uint8)
    shifts = np.zeros((nframes, 2), np.int32)  # shift of frame i relative to frame i-1 (dx, dy); (0, 0) at a scene cut
    rng = np.random.default_rng(seed)
    per = max(1, min(per_base, nframes))
    nbase = (nframes + per - 1) // per
    for i in range(nframes):
        if i % per:
            shifts[i] = (int(rng.integers(-6, 7)), int(rng.integers(-4, 5)))

    def one_scene(b):
        cur = textured_frame(W, H, seed=seed * 100 + b)
        for k in range(per):
            i = b * per + k
            if i >= nframes:
                break
            if k > 0:
                cur = shifted_frame(cur, int(shifts[i, 0]), int(shifts[i, 1]), seed=seed * 1000 + i)
            frames[i] = cur

    with ThreadPoolExecutor(max_workers=min(nbase, usable_cores())) as ex:
        list(ex.map(one_scene, range(nbase)))
    return frames, shifts


def usable_cores():
    """Host threads this process may really use: the affinity mask, capped by the cgroup CPU quota if there is one."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    q = cgroup_cpu_quota()
    if q:
        n = max(1, min(n, int(q + 0.5)))
    return n


def pin_to_gpu_numa_node(torch, local_rank):
    """Restrict this rank's host threads to the CPUs of the NUMA node its GPU hangs off (sysfs local_cpulist of the PCI
    device): pinned-memory uploads and the ctypes worker threads then stay on the socket with the PCIe root port.  Best
    effort: returns a short description, never fails."""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id)
        txt = open("/sys/bus/pci/devices/%s/local_cpulist" % bdf).read().strip()
        cpus = set()
        for part in txt.split(","):
            a, _, b = part.partition("-")
            cpus |= set(range(int(a), int(b or a) + 1))
        cpus &= set(os.sched_getaffinity(0))
        if not cpus:
            return "no local cpus in the affinity mask"
        os.sched_setaffinity(0, cpus)
        return "%s: %d cpus (%s)" % (bdf, len(cpus), txt)
    except Exception as e:
        return "not pinned (%r)" % (e,)


def cgroup_cpu_quota():
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    return float(txt[0]) / float(txt[1])
            else:
                quota = float(txt[0])
                if quota > 0:
                    return quota / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read().split()[0])
        except Exception:
            pass
    return None


WORKLOAD = "configs[1]: 1920x1080 u8 stream, 2000 kp, 8 levels, scale 1.2, frame-to-frame SearchByProjection th=15"
SEMANTICS = {"blur_engine": "OpenCV 2.4 integer GaussianBlur (taps 18,34,49,55,49,34,18 per pass, /65536 half-even), pinned to "
                            "cv2.sepFilter2D with those taps, NOT to cv2.GaussianBlur of OpenCV >= 3.4",
             "retain_best_tie_rule": "canonical: top-n by response, ties at the cut by earlier raster position; differs from "
                                     "libstdc++ nth_element on 17 of 1000 keypoints at 640x480 (same score multiset)"}


def config_dict(args):
    """Identical for both arms (`--impl orbfe` and `--impl reference`): the driver compares them."""
    ab = algorithmic_bytes()
    return {"workload": WORKLOAD, "frames_per_step_per_gpu": args.frames, "batch": args.batch, "passes_per_step": args.repeat,
            "parallelism": "frames sharded one stream per GPU, no data-path collective",
            "l2": "a step's %d distinct input frames are %.0f MB (+ %.0f MB of pyramids per batch): larger than L2 (126 MB)"
                  % (args.frames, args.frames * W * H / 1e6, args.batch * 2 * ab["P"] / 1e6),
            "semantics": SEMANTICS}


def tcw_for_shift(dx, dy):
    """Camera translation that moves every point at depth DEPTH by (dx, dy) pixels."""
    T = np.zeros((3, 4), np.float32)
    T[0, 0] = T[1, 1] = T[2, 2] = 1.0
    T[0, 3] = dx * DEPTH / FX
    T[1, 3] = dy * DEPTH / FY
    return T


def backproject(kps):
    w = np.empty((len(kps), 3), np.float32)
    w[:, 0] = (kps["x"] - np.float32(CX)) / np.float32(FX) * np.float32(DEPTH)
    w[:, 1] = (kps["y"] - np.float32(CY)) / np.float32(FY) * np.float32(DEPTH)
    w[:, 2] = DEPTH
    return w


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    # the sampler runs from before the warm-up (nvidia-smi needs ~1 s to start); only samples whose arrival time
    # falls inside [t_begin, t_end] (the timed region) are used

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []
        self.t_begin = None
        self.t_end = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        inside = [ln for t, ln in self.lines if self.t_begin is not None and self.t_begin <= t <= (self.t_end or 1e30)]
        scope = "timed region"
        if not inside:
            inside, scope = [ln for _, ln in self.lines], "whole run (timed region shorter than the sampling period)"
        for ln in inside:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "scope": scope}


# ------------------------------------------------------------------------------------------------
# CPU side (oracle port of the reference path): the only place bench.py executes oracle/
# ------------------------------------------------------------------------------------------------
def cpu_reference_pass(frames, shifts, threads, reps=None):
    """Oracle extract + SearchByProjection over consecutive frames with `threads` host threads (one frame per task).
    The frame list is repeated until every thread has at least two extraction tasks (with fewer tasks than threads the
    machine would sit half idle and the baseline would be understated).  Only the calls into the C oracle are timed:
    ORBextractor::operator() per frame, then ORBmatcher::SearchByProjection per pair; building the Frame objects in
    between (keypoint grid, Frame.cc:56-125 -- the reference does that in Frame's constructor, outside both classes)
    is not.  Returns (keypoints processed, seconds, extract seconds, match seconds)."""
    import oracle as O
    from concurrent.futures import ThreadPoolExecutor
    n = len(frames)
    reps = reps or max(1, -(-2 * threads // n))
    tasks = n * reps

    def extract_one(t):
        p = O.make_params(NFEAT, SCALE, NLEVELS, 1, FAST_TH)
        rc, k, d, _ = O.extract(p, frames[t % n])
        assert rc == 0
        return k, d

    def frame_one(t, feats):
        k, d = feats[t]
        return O.OracleFrame(k, d, W, H, SCALE, NLEVELS), backproject(k), np.ones(len(k), np.uint8), np.zeros(len(k), np.uint8)

    def match_one(t, fr):
        i = t % n
        if i == 0:
            return 0
        (fl, wl, ones, zeros), (fc, _, _, _) = fr[t - 1], fr[t]
        nm, _ = O.search_by_projection_ff(fc, fl, ones, zeros, wl, tcw_for_shift(*shifts[i]), FX, FY, CX, CY, MATCH_TH, True)
        return nm

    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(lambda t: t, range(threads)))          # spin the worker threads up outside the timed region
        t0 = time.perf_counter()
        feats = list(ex.map(extract_one, range(tasks)))
        t1 = time.perf_counter()
        fr = list(ex.map(lambda t: frame_one(t, feats), range(tasks)))   # untimed: Frame construction
        t2 = time.perf_counter()
        list(ex.map(lambda t: match_one(t, fr), range(tasks)))
        t3 = time.perf_counter()
    return sum(len(k) for k, _ in feats), (t1 - t0) + (t3 - t2), t1 - t0, t3 - t2


def cv2_building_blocks(frame, threads):
    """Third CPU line (SURVEY.md 8d): the OpenCV primitives the reference spends its time in, called through python-cv2
    4.13 on one 1080p frame -- 7 x cv2.resize, FAST(20) + NMS on every level (whole level instead of per cell: same
    pixels), 8 x sepFilter2D with the 2.4 integer taps.  A labelled building-block time, NOT the reference pipeline
    (no per-cell logic, retention, orientation or descriptors)."""
    try:
        import cv2
    except Exception as e:
        return {"unavailable": "cv2 import failed: %s" % e}
    from concurrent.futures import ThreadPoolExecutor
    k = (np.array([18, 34, 49, 55, 49, 34, 18], np.float64) / 256.0)
    sizes = level_sizes()
    fast = cv2.FastFeatureDetector_create(FAST_TH, True)

    def one(_):
        lv = [frame]
        for w, h in sizes[1:]:
            lv.append(cv2.resize(lv[-1], (w, h), interpolation=cv2.INTER_LINEAR))
        nk = 0
        for im in lv:
            nk += len(fast.detect(im[13:-13, 13:-13], None))
            cv2.sepFilter2D(im, cv2.CV_8U, k, k, borderType=cv2.BORDER_REFLECT_101)
        return nk

    cv2.setNumThreads(1)
    one(0)
    t0 = time.perf_counter()
    for _ in range(3):
        one(0)
    ms1 = (time.perf_counter() - t0) / 3 * 1e3
    ntask = 2 * threads
    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(lambda t: t, range(threads)))
        t0 = time.perf_counter()
        list(ex.map(one, range(ntask)))
        dt = time.perf_counter() - t0
    return {"what": "python-cv2 %s: 7 resize + whole-level FAST(20)+NMS on 8 levels + 8 sepFilter2D(2.4 taps), one 1080p frame; "
                    "building blocks only, not the reference pipeline" % cv2.__version__,
            "ms_per_frame_1_thread": ms1, "frames_per_s_%d_threads" % threads: ntask / dt}


def cpu_baseline_dict(frames, shifts, steps, warm):
    """The CPU arm: oracle port on all usable host threads + its single-thread figure + parallel efficiency."""
    threads = usable_cores()
    nfr = max(2, min(len(frames), 64))
    fr, sh = frames[:nfr], shifts[:nfr]
    if warm:
        cpu_reference_pass(fr[:2], sh[:2], min(threads, 2), reps=1)
    tot_kp, tot_t, tot_x, tot_m = 0, 0.0, 0.0, 0.0
    for _ in range(max(1, steps)):
        kp, dt, dx, dm = cpu_reference_pass(fr, sh, threads)
        tot_kp += kp; tot_t += dt; tot_x += dx; tot_m += dm
    val = tot_kp / tot_t / 1e6
    kp1, dt1, _, _ = cpu_reference_pass(fr[:4], sh[:4], 1, reps=1)   # the reference's own mode: one Tracking thread
    single = kp1 / dt1 / 1e6
    reps = max(1, -(-2 * threads // nfr))
    d = {"value": val, "unit": "Mkeypoints/s", "cores": threads, "kind": "port",
         "single_thread_value": single, "parallel_efficiency": val / (threads * single) if single > 0 else None,
         "host": {"os_cpu_count": os.cpu_count(), "sched_affinity": len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else None,
                  "cgroup_cpu_quota": cgroup_cpu_quota()},
         "extract_s": tot_x, "match_s": tot_m,
         "sample": "%d distinct 1080p frames repeated to %d extract+match tasks per pass x %d passes, CPU oracle port "
                   "(oracle/liborb_oracle.so, gcc -O3 -march=native; the reference itself needs OpenCV 2.4/ROS and cannot be "
                   "built here) on %d threads, %.1f s timed; Frame construction between extract and match not timed"
                   % (nfr, nfr * reps, max(1, steps), threads, tot_t)}
    try:
        d["cv2_building_blocks"] = cv2_building_blocks(frames[0], threads)
    except Exception as e:   # a labelled extra, never fatal
        d["cv2_building_blocks"] = {"unavailable": repr(e)}
    return d, tot_t / max(1, steps)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    nframes = max(2, min(usable_cores(), 64))
    frames, shifts = make_stream(nframes, seed=7)
    cb, s_per_step = cpu_baseline_dict(frames, shifts, args.steps, args.warmup > 0)
    val = cb["value"]
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Mkeypoints/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": s_per_step * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": config_dict(args),
            "cpu_baseline": cb,
            "e2e": {"value": val, "unit": "Mkeypoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="orbfe", choices=["orbfe", "reference"])
    ap.add_argument("--frames", type=int, default=256, help="distinct frames per step per GPU")
    ap.add_argument("--batch", type=int, default=64, help="frames per library call")
    ap.add_argument("--repeat", type=int, default=4, help="passes over the step's frames inside one step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle cross-check of the step's results (ncu runs)")
    ap.add_argument("--workload", default="stream", choices=["stream", "rig8", "dbsweep"],
                    help="stream = BASELINE configs[1] (the headline line); rig8 = configs[3] (one camera per GPU, exchange + cross-camera "
                         "SearchForInitialization); dbsweep = configs[4] (sharded keyframe-database sweep): the last two print their own line")
    ap.add_argument("--slots", type=int, default=8, help="rig8: time steps per exchange")
    ap.add_argument("--groups", type=int, default=10000, help="dbsweep: keyframes in the database")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the keypoints, descriptors and matches the value path returned in its "
                    "last timed step (a fixed sample of %d frames) as DIR/<name>.npy" % DUMP_FRAMES)
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "stream" or args.impl != "orbfe"):
        ap.error("--dump-outputs writes the results of the stream workload of --impl orbfe")
    if args.workload != "stream" and args.impl == "orbfe":
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import multi_gpu
        ctx = multi_gpu._setup()
        out = (multi_gpu.run_rig if args.workload == "rig8" else multi_gpu.run_dbsweep)(args, ctx)
        if ctx[3] == 0:
            print(json.dumps(out))
        if ctx[2] > 1:
            ctx[1].destroy_process_group()
        return 0
    args.frames = max(args.batch, args.frames // args.batch * args.batch)
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import orb_slam_b200 as fe
    from orb_slam_b200 import matching as M

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: liborbfe has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    numa = pin_to_gpu_numa_node(torch, local_rank) if world > 1 else "single rank: not pinned"

    B = args.batch
    NB = args.frames // B                      # batches per pass
    SUB = NB * args.repeat                     # library calls (sub-steps) per step
    frames_np, shifts = make_stream(args.frames, seed=11 + rank)
    # a pass wraps around: frame 0 follows frame F-1 of the previous pass (a scene cut: shift 0, no true matches)
    h_frames = torch.from_numpy(frames_np).pin_memory()                 # pinned host input (e2e path)
    d_frames = torch.from_numpy(frames_np).to(dev)                      # resident input (value path)

    ex = fe.ORBextractor(NFEAT, SCALE, NLEVELS, fe.FAST_SCORE, FAST_TH, device=local_rank)
    mt = fe.ORBmatcher(0.9, True, device=local_rank)
    ex.set_profiling(True)
    # a dedicated (non-default) stream: the library's kernels and torch's async copies share it
    stream = torch.cuda.Stream(device=dev)
    Tcws = [tcw_for_shift(*shifts[i]) for i in range(args.frames)]
    stage_acc, stage_n = {}, [0]
    kp_total = [0]
    launches = [0]
    host_t = {"extract_call": 0.0, "e2e_extract_call": 0.0, "match_call": 0.0, "views": 0.0, "n": 0}
    ones_u8, zeros_u8 = np.ones(NFEAT, np.uint8), np.zeros(NFEAT, np.uint8)
    checks = {"device": None, "e2e": None}    # last finished sub-step of each path, for the oracle cross-check
    # --dump-outputs: the sampled frames' results, filled while the last timed step finishes its batches
    dump_frames = np.sort(np.random.default_rng(0).choice(args.frames, min(args.frames, DUMP_FRAMES), replace=False))
    dump = {"keypoints": np.zeros((len(dump_frames), NFEAT, 7), np.float32),
            "descriptors": np.zeros((len(dump_frames), NFEAT, 32), np.float32),
            "keypoint_counts": np.full(len(dump_frames), -1, np.float32),
            "matches": np.zeros((len(dump_frames), NFEAT), np.float32),
            "match_counts": np.zeros(len(dump_frames), np.float32),
            "frame_index": dump_frames.astype(np.float32)} if args.dump_outputs and rank == 0 else None

    Tcws_arr = np.ascontiguousarray(np.stack(Tcws).reshape(args.frames, 12), np.float32)
    ones_ptr, zeros_ptr = np.uint64(ones_u8.ctypes.data), np.uint64(zeros_u8.ctypes.data)

    def prepare_views(kps_a, desc_a, cnt_a):
        """Frame views + synthetic map points of one batch's host results (array operations over the whole batch: this glue
        stands for the reference's C++ Frame construction and must not be what the pipeline waits for), plus a private
        copy of the batch's last frame (the Last frame of the next batch's first pair; the pinned buffers are reused)."""
        t0 = time.perf_counter()
        batch = M.FrameViewBatch(kps_a, desc_a, cnt_a, W, H, SCALE, NLEVELS)
        wpts = np.empty((B, NFEAT, 3), np.float32)            # same float32 ops as backproject()
        wpts[:, :, 0] = (kps_a["x"] - np.float32(CX)) / np.float32(FX) * np.float32(DEPTH)
        wpts[:, :, 1] = (kps_a["y"] - np.float32(CY)) / np.float32(FY) * np.float32(DEPTH)
        wpts[:, :, 2] = DEPTH
        tail_view, tail_keep = batch.tail()
        tail = (tail_view, wpts[B - 1].copy(), tail_keep)
        host_t["views"] += time.perf_counter() - t0
        return batch, wpts, tail

    def match_step(sb, prepared, prev_prepared, matcher):
        batch, world_cur, tail = prepared
        t1 = time.perf_counter()
        pv, pw, _keep = prev_prepared[2] if prev_prepared is not None else tail
        views_last = np.concatenate([pv, batch.views[:-1]])
        wrows = M.row_pointers(world_cur)
        world_ptrs = np.concatenate([np.array([pw.ctypes.data], np.uint64), wrows[:-1]])
        mp = np.full((B, NFEAT), -1, np.int32)
        nm = M.search_by_projection_views(matcher, batch.views, views_last, np.full(B, ones_ptr, np.uint64), np.full(B, zeros_ptr, np.uint64),
                                          world_ptrs, Tcws_arr[sb * B:(sb + 1) * B], FX, FY, CX, CY, MATCH_TH, mp)
        host_t["match_call"] += time.perf_counter() - t1
        host_t["n"] += 1
        cn = batch.counts
        checks["e2e"] = (sb, [batch.kps[i, :cn[i]].copy() for i in range(4)], [batch.desc[i, :cn[i]].copy() for i in range(4)],
                         [mp[i].copy() for i in range(4)])
        return int(nm.sum())

    stage_cnt = {}

    def collect_stages():
        # per-stage sums AND occurrence counts: the per-batch figure is sum / count, whatever number of intervals came back
        for name, ms in ex.stage_times():
            stage_acc[name] = stage_acc.get(name, 0.0) + ms
            stage_cnt[name] = stage_cnt.get(name, 0) + 1
        stage_n[0] += 1

    # ---- device-resident pipeline (value path).  Two buffer sets: while batch t is matched and read back on
    # stream_m, batch t+1 is already being extracted on stream_x.  Slot B of a set holds the previous batch's last frame.
    def make_set():
        S = {}
        S["kps"] = torch.zeros((B + 1, NFEAT, 28), dtype=torch.uint8, device=dev)
        S["desc"] = torch.zeros((B + 1, NFEAT, 32), dtype=torch.uint8, device=dev)
        S["cnt"] = torch.zeros((B + 1,), dtype=torch.int32, device=dev)
        S["world"] = torch.zeros((B + 1, NFEAT, 3), dtype=torch.float32, device=dev)
        S["mp"] = torch.empty((B, NFEAT), dtype=torch.int32, device=dev)
        S["nm"] = torch.zeros((B,), dtype=torch.int32, device=dev)
        S["kxy"] = S["kps"].view(torch.float32).view(B + 1, NFEAT, 7)
        S["h_kps"] = torch.empty((B, NFEAT, 28), dtype=torch.uint8).pin_memory()
        S["h_desc"] = torch.empty((B, NFEAT, 32), dtype=torch.uint8).pin_memory()
        S["h_cnt"] = torch.zeros((B,), dtype=torch.int32).pin_memory()
        S["h_mp"] = torch.empty((B, NFEAT), dtype=torch.int32).pin_memory()
        S["h_nm"] = torch.zeros((B,), dtype=torch.int32).pin_memory()
        S["ev_x"] = torch.cuda.Event()
        S["ev_done"] = torch.cuda.Event()
        S["sb"] = -1
        return S

    dsets = [make_set(), make_set()]
    d_flags = torch.ones((B + 1, NFEAT), dtype=torch.uint8, device=dev)   # every feature carries a map point
    d_T = torch.from_numpy(np.stack(Tcws).reshape(args.frames, 12)).to(dev)
    d_cur = torch.arange(0, B, dtype=torch.int32, device=dev)
    d_last = torch.tensor([B] + list(range(0, B - 1)), dtype=torch.int32, device=dev)
    stream_m = torch.cuda.Stream(device=dev, priority=-1)   # the short matcher kernel goes first when SMs free up
    stream_b = stream_m
    dev_state = {"step": 0, "capture_from": None}

    def enqueue_device_step():
        st = dev_state["step"]
        sb = st % NB
        S, Pv = dsets[st & 1], dsets[(st - 1) & 1]
        with torch.cuda.stream(stream):
            stream.wait_event(S["ev_done"])          # the set's previous results have left the device
            ex.extract_batch_device(d_frames.data_ptr() + sb * B * W * H, W, H, W, W * H, B, S["kps"].data_ptr(), S["desc"].data_ptr(),
                                    S["cnt"].data_ptr(), stream.cuda_stream)
            # synthetic map points: back-project every keypoint at depth DEPTH (same float32 ops as backproject())
            S["world"][:B, :, 0] = (S["kxy"][:B, :, 0] - CX) / FX * DEPTH
            S["world"][:B, :, 1] = (S["kxy"][:B, :, 1] - CY) / FY * DEPTH
            S["world"][:B, :, 2] = DEPTH
            S["ev_x"].record(stream)
        with torch.cuda.stream(stream_m):
            stream_m.wait_event(S["ev_x"])
            # slot B <- last frame of the previous batch (extracted earlier on `stream`, matched earlier on stream_m)
            S["kps"][B].copy_(Pv["kps"][B - 1]); S["desc"][B].copy_(Pv["desc"][B - 1])
            S["cnt"][B:B + 1].copy_(Pv["cnt"][B - 1:B]); S["world"][B].copy_(Pv["world"][B - 1])
            S["mp"].fill_(-1)
            M.search_by_projection_device(mt, B, S["kps"].data_ptr(), S["desc"].data_ptr(), S["cnt"].data_ptr(), NFEAT,
                                          d_cur.data_ptr(), d_last.data_ptr(), S["world"].data_ptr(), d_flags.data_ptr(),
                                          d_T.data_ptr() + sb * B * 48, W, H, SCALE, NLEVELS, FX, FY, CX, CY, MATCH_TH,
                                          S["mp"].data_ptr(), S["nm"].data_ptr(), stream_m.cuda_stream)
            S["h_cnt"].copy_(S["cnt"][:B], non_blocking=True)
            S["h_nm"].copy_(S["nm"], non_blocking=True)
            S["h_kps"].copy_(S["kps"][:B], non_blocking=True)
            S["h_desc"].copy_(S["desc"][:B], non_blocking=True)
            S["h_mp"].copy_(S["mp"], non_blocking=True)
            S["ev_done"].record(stream_m)
        S["sb"] = sb
        S["capture"] = dump is not None and dev_state["capture_from"] is not None and st >= dev_state["capture_from"]
        launches[0] += ex.last_launches() + 1
        dev_state["step"] = st + 1
        return S

    def finish_device_step(S):
        S["ev_done"].synchronize()
        kp_total[0] += int(S["h_cnt"].numpy().sum())
        checks["device"] = S
        if S["capture"]:
            capture_batch(S)
        return int(S["h_nm"].numpy().sum())

    def capture_batch(S):
        """--dump-outputs: the sampled frames of this batch, as a caller of the value path receives them (rows past a frame's
        keypoint count are not part of its result and stay zero)"""
        lo = S["sb"] * B
        kd = S["h_kps"].numpy().view(fe.KP_DTYPE).reshape(B, NFEAT)
        for j in np.flatnonzero((dump_frames >= lo) & (dump_frames < lo + B)):
            i, n = int(dump_frames[j]) - lo, int(S["h_cnt"].numpy()[int(dump_frames[j]) - lo])
            dump["keypoints"][j] = 0
            dump["descriptors"][j] = 0
            for c, name in enumerate(fe.KP_DTYPE.names):
                dump["keypoints"][j, :n, c] = kd[i, :n][name]
            dump["descriptors"][j, :n] = S["h_desc"].numpy()[i, :n]
            dump["keypoint_counts"][j] = n
            dump["matches"][j] = S["h_mp"].numpy()[i]
            dump["match_counts"][j] = S["h_nm"].numpy()[i]

    def run_device(steps, capture_last=False):
        """`steps` steps of SUB batches; with capture_last the batches of the last step fill `dump`"""
        t0 = time.perf_counter()
        dev_state["capture_from"] = dev_state["step"] + (steps - 1) * SUB if capture_last else None
        nm, pending = 0, None
        for _ in range(steps * SUB):
            S = enqueue_device_step()
            if pending is not None:
                nm += finish_device_step(pending)
            pending = S
        nm += finish_device_step(pending)
        stream.synchronize()
        collect_stages()
        host_t["extract_call"] += time.perf_counter() - t0
        return nm

    # ---- e2e: host buffers in, host results out.  A stream of frames is processed as a software pipeline over the
    # public C-ABI calls only: two extractor handles (each with its own device buffers and streams) alternate batches on
    # two host threads, so the upload of batch t+1 overlaps the kernels of batch t and there is no bubble at a call
    # boundary; frame views (the host-side Frame objects of the reference) are built on their own worker threads and
    # a last thread matches finished batches in order (orbfe_search_by_projection_frames on host views).
    # ctypes releases the GIL inside the calls.  Outputs rotate through four pinned buffer sets.
    from concurrent.futures import ThreadPoolExecutor
    NEX = max(1, int(os.environ.get("ORBFE_E2E_EXTRACTORS", "3")))   # extractor handles in flight
    os.environ.setdefault("ORBFE_CHUNKS", "2")   # upload chunks per host batch: with three handles in flight two chunks measured best
    NMATCH = max(1, int(os.environ.get("ORBFE_E2E_MATCHERS", "3")))  # matcher handles in flight (C++ driver)
    NBUF = NEX + NMATCH
    e2e_bufs = []
    for _ in range(NBUF):
        hk = torch.empty((B, NFEAT, 28), dtype=torch.uint8).pin_memory()
        hd = torch.empty((B, NFEAT, 32), dtype=torch.uint8).pin_memory()
        hc = torch.empty((B,), dtype=torch.int32).pin_memory()
        e2e_bufs.append((hk, hd, hc, hk.numpy().view(fe.KP_DTYPE).reshape(B, NFEAT), hd.numpy(), hc.numpy()))
    USE_PY_E2E = os.environ.get("ORBFE_E2E_PY") == "1"           # Python-thread pipeline instead of the C++ driver (below)
    e2e_ex = [ex] + [fe.ORBextractor(NFEAT, SCALE, NLEVELS, fe.FAST_SCORE, FAST_TH, device=local_rank) for _ in range(NEX - 1 if USE_PY_E2E else 0)]
    e2e_ex_pool = [ThreadPoolExecutor(max_workers=1) for _ in range(NEX)]
    E2E_MODE = int(os.environ.get("ORBFE_E2E_BATCH_MODE", "0"))   # measured: chunked 28.7 vs phased 26.8 Mkp/s with two handles
    e2e_mt = (mt, fe.ORBmatcher(0.9, True, device=local_rank)) if USE_PY_E2E else (mt,)
    e2e_match_pool = (ThreadPoolExecutor(max_workers=1), ThreadPoolExecutor(max_workers=1))
    e2e_views_pool = ThreadPoolExecutor(max_workers=2)
    e2e_state = {"step": 0}

    def extract_step(st):
        t0 = time.perf_counter()
        x = e2e_ex[st % NEX]
        x.set_batch_mode(E2E_MODE)
        hk, hd, hc, _, _, c_np = e2e_bufs[st % NBUF]
        x.extract_batch_ptr(h_frames.data_ptr() + (st % NB) * B * W * H, W, H, W, W * H, B, hk.data_ptr(), hd.data_ptr(), NFEAT,
                            hc.data_ptr())
        host_t["e2e_extract_call"] += time.perf_counter() - t0
        return x.last_launches(), int(c_np.sum())

    def run_e2e_python(steps):
        nm = 0
        ex_futs, m_futs, v_futs = {}, {}, {}
        s0 = e2e_state["step"]
        nsub = steps * SUB

        def finish_extract(st):
            nl, nk = ex_futs.pop(st).result()
            launches[0] += nl
            kp_total[0] += nk
            _, _, _, k_np, d_np, c_np = e2e_bufs[st % NBUF]
            vf = e2e_views_pool.submit(prepare_views, k_np, d_np, c_np)   # frame views: a stage of its own
            pf = v_futs.get(st - 1)
            v_futs[st] = vf
            v_futs.pop(st - 2, None)
            # two matcher handles alternate so that the queueing latency of one call hides behind the other
            m_futs[st] = e2e_match_pool[st & 1].submit(
                lambda f=vf, p=pf, mm=e2e_mt[st & 1], sb=st % NB: match_step(sb, f.result(), p.result() if p is not None else None, mm))

        for st in range(s0, s0 + nsub):
            if st - (NBUF - 1) in m_futs:             # buffer set st % NBUF was last used by batch st - NBUF
                nm += m_futs.pop(st - (NBUF - 1)).result()
            ex_futs[st] = e2e_ex_pool[st % NEX].submit(extract_step, st)
            if st - s0 >= NEX - 1:
                finish_extract(st - (NEX - 1))
        for st in sorted(ex_futs):
            finish_extract(st)
        for st in sorted(m_futs):
            nm += m_futs[st].result()
        e2e_state["step"] = s0 + nsub
        return nm

    # The same pipeline on C++ threads (tools/e2e_driver.cpp -> orb_slam_b200/libe2e_driver.so; default): a C++ host -- what the
    # reference's Tracking thread is -- calling orbfe_extract_batch / orbfe_search_by_projection_frames of liborbfe.so, nothing
    # else.  The Python-thread version above is kept behind ORBFE_E2E_PY=1: its GIL hand-offs cost more than the calls themselves.
    import ctypes as C
    drv = {"d": None, "mh2d": 0, "md2h": 0}
    if not USE_PY_E2E:
        from orb_slam_b200.stream_driver import StreamDriver
        drv["d"] = StreamDriver(W, H, NFEAT, NLEVELS, SCALE, FAST_TH, B, NB, NEX, NMATCH, local_rank, FX, FY, CX, CY, DEPTH, MATCH_TH,
                                h_frames.data_ptr(), Tcws_arr, [b_[0].data_ptr() for b_ in e2e_bufs], [b_[1].data_ptr() for b_ in e2e_bufs],
                                [b_[2].data_ptr() for b_ in e2e_bufs])

    def run_e2e_driver(steps):
        r = drv["d"].run(steps * SUB)
        kp_total[0] += r["keypoints"]
        launches[0] += r["extract_launches"] + r["match_launches"]
        drv["mh2d"] += r["match_h2d"]
        drv["md2h"] += r["match_d2h"]
        host_t["e2e_extract_call"] += r["extract_s"]; host_t["views"] += r["views_s"]; host_t["match_call"] += r["match_s"]
        host_t["n"] += steps * SUB
        # the last matched batch, for the oracle cross-check: its keypoints / descriptors still sit in their pinned output set
        st = int(r["last_batch"])
        _, _, _, k_np, d_np, c_np = e2e_bufs[st % NBUF]
        mp4 = drv["d"].last_matches()
        checks["e2e"] = (st % NB, [k_np[i, :c_np[i]].copy() for i in range(4)], [d_np[i, :c_np[i]].copy() for i in range(4)], list(mp4))
        return int(r["matches"])

    run_e2e = run_e2e_python if USE_PY_E2E else run_e2e_driver

    def timed(run_fn, steps):
        kp_total[0] = 0
        launches[0] = 0
        c0 = [sum(x) for x in zip(*(m_.counters() for m_ in e2e_mt))]
        d0 = (drv["mh2d"], drv["md2h"])
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        nm = run_fn(steps)
        stream.wait_stream(stream_b)
        e1.record(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = max(e0.elapsed_time(e1), 0.0)
        c1 = [sum(x) for x in zip(*(m_.counters() for m_ in e2e_mt))]
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device=dev)
        k = torch.tensor([kp_total[0], nm], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(k, op=dist.ReduceOp.SUM)
            dist.barrier()
        return {"ms": float(t[0]), "wall_ms": float(t[1]), "kp": float(k[0]), "matches": float(k[1]),
                "launches": launches[0] + (c1[2] - c0[2]), "mh2d": c1[0] - c0[0] + drv["mh2d"] - d0[0], "md2h": c1[1] - c0[1] + drv["md2h"] - d0[1]}

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    run_device(args.warmup)
    ex.set_profiling(False)          # stage events only during the device-resident timed region
    run_e2e(args.warmup)
    ex.set_profiling(True)
    ex.stage_times()                 # flush
    stage_acc.clear()
    stage_cnt.clear()
    stage_n[0] = 0

    sampler.t_begin = time.perf_counter()
    r_dev = timed(lambda steps: run_device(steps, capture_last=dump is not None), args.steps)
    stages = {k: v / max(stage_cnt.get(k, 1), 1) * SUB for k, v in stage_acc.items()}   # ms per step (= SUB library calls)
    if rank == 0 and stage_cnt and min(stage_cnt.values()) != args.steps * SUB:
        sys.stderr.write("bench: stage intervals read back for %s of %d batches\n" % (sorted(set(stage_cnt.values())), args.steps * SUB))
    ex.set_profiling(False)
    r_e2e = timed(run_e2e, args.steps)
    sampler.t_end = time.perf_counter()
    clocks = sampler.stop() if rank == 0 else None

    # stage times once more with the extractor alone on the GPU (in the timed region above the matcher of the
    # previous batch shares the SMs with whatever stage is running): a stable figure for kernel-to-kernel comparisons
    ex.set_profiling(True)
    ex.stage_times()
    S0 = dsets[0]
    iso_acc, iso_n = {}, 8
    for i in range(iso_n):
        ex.extract_batch_device(d_frames.data_ptr() + (i % NB) * B * W * H, W, H, W, W * H, B, S0["kps"].data_ptr(),
                                S0["desc"].data_ptr(), S0["cnt"].data_ptr(), stream.cuda_stream)
    stream.synchronize()
    for name, ms in ex.stage_times():
        iso_acc[name] = iso_acc.get(name, 0.0) + ms / iso_n       # ms per batch of B frames
    ex.set_profiling(False)

    # latency of the reference's own usage pattern: one frame per call, host image in, host keypoints/descriptors out
    # (ORBextractor::operator(), src/ORBextractor.cc:718-779), nothing else on the GPU
    lat = []
    hk1, hd1, hc1 = e2e_bufs[0][0], e2e_bufs[0][1], e2e_bufs[0][2]
    for i in range(25):
        t0 = time.perf_counter()
        ex.extract_batch_ptr(h_frames.data_ptr() + (i % args.frames) * W * H, W, H, W, W * H, 1, hk1.data_ptr(), hd1.data_ptr(), NFEAT,
                             hc1.data_ptr())
        lat.append((time.perf_counter() - t0) * 1e3)
    single_ms = float(np.median(lat[5:]))

    # ---- oracle cross-check of what the timed region produced (outside it; rank 0 only; the one place besides the CPU arm
    # where bench.py touches oracle/): keypoints + descriptors of the first four frames of the last batch of each path,
    # and the match vectors of the three pairs among them, must equal the CPU oracle's on the same frames
    parity = None
    if rank == 0 and not args.no_parity:
        import oracle as O
        p = O.make_params(NFEAT, SCALE, NLEVELS, 1, FAST_TH)
        parity = {"frames": 0, "pairs": 0, "paths": []}

        def check(tag, sb, kps4, desc4, mp4):
            of = []
            for i in range(4):
                rc, ok, od, _ = O.extract(p, frames_np[sb * B + i])
                assert rc == 0, rc
                gk = kps4[i]
                assert len(gk) == len(ok), (tag, sb, i, len(gk), len(ok))
                for name in ("x", "y", "size", "response", "octave", "class_id"):
                    assert np.array_equal(gk[name], ok[name]), (tag, sb, i, name)
                assert np.max(np.abs(gk["angle"] - ok["angle"]), initial=0.0) <= 1e-4, (tag, sb, i, "angle")
                assert np.array_equal(desc4[i], od), (tag, sb, i, "descriptors")
                of.append((O.OracleFrame(ok, od, W, H, SCALE, NLEVELS), ok))
                parity["frames"] += 1
            for i in range(1, 4):
                (fc, _), (fl, kl) = of[i], of[i - 1]
                n_o, mp_o = O.search_by_projection_ff(fc, fl, ones_u8[:fl.n], zeros_u8[:fl.n], backproject(kl), Tcws[sb * B + i],
                                                      FX, FY, CX, CY, MATCH_TH, True)
                assert np.array_equal(mp4[i][:fc.n], mp_o), (tag, sb, i, "matches")
                parity["pairs"] += 1
            parity["paths"].append(tag)

        S = checks["device"]
        cn = S["h_cnt"].numpy()
        kd = S["h_kps"].numpy().view(fe.KP_DTYPE).reshape(B, NFEAT)
        check("value: orbfe_extract_batch_device + orbfe_search_by_projection_device", S["sb"],
              [kd[i, :cn[i]] for i in range(4)], [S["h_desc"].numpy()[i, :cn[i]] for i in range(4)],
              [S["h_mp"].numpy()[i] for i in range(4)])
        sb, k4, d4, m4 = checks["e2e"]
        check("e2e: orbfe_extract_batch + orbfe_search_by_projection_frames", sb, k4, d4, m4)

    if rank == 0:
        ab = algorithmic_bytes()
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        # dominant kernel of the extract pipeline by measured stage time; per launch = per batch of B frames
        kernel_stages = {k: v / SUB for k, v in stages.items() if k not in ("ingest", "h2d", "d2h")}
        dom = max(kernel_stages, key=kernel_stages.get) if kernel_stages else None
        dom_bytes = {"fast_nms": ab["fast_read"], "blur7": ab["blur"], "pyramid": ab["resize"]}.get(dom, ab["total"]) * B
        dom_ms = kernel_stages.get(dom, 0.0) if dom else 0.0
        achieved = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
        ext_ms = sum(kernel_stages.values())
        traffic, alu = None, None
        try:  # DRAM bytes + ALU-pipe instructions of the dominant kernel from the committed ncu capture, scaled to B frames
            tj = json.load(open(os.path.join(ROOT, "profiles", "fast_nms_ncu.json")))
            if dom == "fast_nms":
                traffic = (tj["dram_bytes_read"] + tj["dram_bytes_write"]) / tj["frames_in_launch"] * B
                # the kernel executes the same ALU-pipe instructions per frame here as under ncu, so its pipe utilisation
                # scales with the ratio of the per-frame durations: frac_live = frac_ncu * t_ncu / t_live
                t_ncu = tj["duration_us"] * 1e-3 / tj["frames_in_launch"]          # ms per frame under ncu
                util_hw = tj["alu_pipe_pct_of_peak"] / 100.0 * t_ncu / (dom_ms / B)   # of the hardware peak (64 /clk/SM)
                a = util_hw * tj["alu_peak_hw_thread_inst_per_clk_sm"]
                scale_t = t_ncu / (dom_ms / B)
                alu = {"achieved": a, "peak": tj["alu_peak_measured_thread_inst_per_clk_sm"],
                       "unit": "ALU-pipe thread-instructions/clk/SM", "frac": a / tj["alu_peak_measured_thread_inst_per_clk_sm"],
                       "peak_source": "tools/ubench_alu.cu on B200 (profiles/r2_ubench_alu.txt): 58.7 (VIMNMX3 / VIMNMX / PRMT / LOP3 share one "
                                      "16-lane pipe per SM sub-partition; hardware peak 64)",
                       "issue_slots_used": tj.get("issue_active_pct", 0.0) / 100.0 * scale_t,
                       "fma_pipe_frac_of_hw_peak": tj.get("fma_pipe_pct_of_peak", 0.0) / 100.0 * scale_t,
                       "issue_note": "warp-instructions issued per cycle per scheduler; the same microbenchmark measures 0.63-0.68 as the most a "
                                     "mix of ALU-pipe and FMA-pipe instructions issues on this SM, 0.46 for ALU-pipe instructions alone: the "
                                     "kernel moved its 2-input min/max pairs to the FMA pipe (exact fp16-subnormal HFMA2) until issue, not a pipe, binds",
                       "how": "ncu sm__inst_executed_pipe_alu %.1f%% of peak, issue active %.1f%%, at %.1f us per frame, scaled by the live per-frame time"
                              % (tj["alu_pipe_pct_of_peak"], tj.get("issue_active_pct", 0.0), t_ncu * 1e3), "source": tj.get("source")}
        except Exception:
            pass
        roof = {"bound": "alu" if alu else "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak if peak else None, "traffic": traffic, "peak_source": peak_src,
                "note": "achieved/peak/frac are the HBM roofline the metric is quoted against; fast_nms is bound by instruction issue "
                        "(integer ALU pipe + FMA pipe, the `alu` entry), not by memory: see profiles/README.md",
                "alu": alu,
                "algorithmic_bytes_per_launch": dom_bytes, "launch_ms": dom_ms, "frames_per_launch": B,
                "extract_all_kernels": {"algorithmic_bytes": ab["total"] * B, "ms": ext_ms,
                                        "achieved": ab["total"] * B / (ext_ms * 1e-3) / 1e9 if ext_ms > 0 else 0.0,
                                        "frac": ab["total"] * B / (ext_ms * 1e-3) / 1e9 / peak if ext_ms > 0 and peak else None},
                "stage_ms_per_batch": {k: v / SUB for k, v in stages.items()}, "stage_ms_per_batch_extractor_alone": iso_acc}
        value = r_dev["kp"] / (r_dev["ms"] * 1e-3) / 1e6
        e2e_val = r_e2e["kp"] / (r_e2e["ms"] * 1e-3) / 1e6
        line = {"metric": METRIC, "value": value, "unit": "Mkeypoints/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": r_dev["ms"] / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config_dict(args),
                "e2e": {"value": e2e_val, "unit": "Mkeypoints/s", "ms_per_step": r_e2e["ms"] / args.steps,
                        "pipeline": ("python threads (ORBFE_E2E_PY=1)" if USE_PY_E2E else "C++ threads over the public C-ABI (tools/e2e_driver.cpp)") +
                                    ": %d extractor handles, %d matcher handles, %s upload chunks per batch; pinned host frames in, host keypoints / "
                                    "descriptors / matches out" % (NEX, NMATCH, os.environ.get("ORBFE_CHUNKS", "4")),
                        # whole job: every rank moves the same amount
                        "h2d_bytes_per_step": world * (SUB * B * W * H + r_e2e["mh2d"] // args.steps),
                        "d2h_bytes_per_step": world * (SUB * B * (NFEAT * 60 + 4) + r_e2e["md2h"] // args.steps)},
                "gpu_launches": int(r_dev["launches"]),
                "timed_region_s": {"value": r_dev["ms"] * 1e-3, "e2e": r_e2e["ms"] * 1e-3},
                "matches_per_step": r_dev["matches"] / args.steps / world,
                "keypoints_per_step": r_dev["kp"] / args.steps,
                "wall_ms_per_step": r_dev["wall_ms"] / args.steps,
                "host_ms_per_batch": {k: 1e3 * v / max(host_t["n"], 1) for k, v in host_t.items() if k != "n"},
                "single_frame_latency_ms": single_ms, "host_numa_pinning_rank0": numa,
                "parity_checked": parity,
                "roofline": roof, "clocks": clocks}
        if not args.no_cpu_baseline:
            line["cpu_baseline"], _ = cpu_baseline_dict(frames_np, shifts, 1, True)
        if dump is not None:
            assert (dump["keypoint_counts"] >= 0).all(), "--dump-outputs: a sampled frame was not produced by the last step"
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dump.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        print(json.dumps(line))
    if drv["d"]:
        drv["d"].close()
    for x in e2e_ex:
        x.close()
    for m_ in e2e_mt:
        m_.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
