#!/usr/bin/env python
"""bench.py -- frames/s of the aruco_detect hot path (detect + pose) on BASELINE.json's config C2.

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA path through the C-ABI)
  python bench.py --impl reference --gpus N --steps K ...   the reference's CPU path (cv2) on host cores
  python bench.py ... --dump-outputs DIR                    also write the last timed step's results to DIR/<name>.npy

A "step" is one pass of the hot path over one batch of synthetic 1920x1080 frames (16 markers of
DICT_6X6_250 each): BGR8 frames -> ids, corners, rvec/tvec, quaternion, image/object error, area,
followed by the per-camera fiducial_slam map update of those messages (and, for N > 1, one NCCL
all-gather + deterministic merge of the per-rank map tables).  Frames shard one stream per GPU,
weak scaling, no collective on the detect/pose path.

  value  : frames/s, whole job, frames already resident in HBM when the timed region starts
  e2e    : frames/s through the same C-ABI call with pinned HOST frames (H2D of every frame and D2H
           of every result inside the timed region)
  roofline: the threshold kernel (the HBM-bound stage BASELINE.json's metric names): algorithmic
           bytes 3*W*H + n_scales*W*H/8 per frame (SURVEY 8d) / its CUDA-event time, vs the measured
           copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline: the same frames through cv2's ArucoDetector + solvePnP + projectPoints (the OpenCV
           calls of aruco_detect.cpp:350,247,210) on this box's host cores, bounded sample
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

WORKLOAD = "C2"  # set by main() from --workload

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FIDUCIAL_LEN = 0.14
DEPTH = int(os.environ.get("FID_BENCH_DEPTH", "2"))            # batches in flight (each takes FRAMES/SLOT of the library's FID_SLOTS chunk slots)
HBM_FALLBACK_GBS = 6650.0
REALIZATIONS = 8   # noise realisations per marker layout of the synthetic stream (a layout costs 0.8 s of numpy to render)
# BASELINE.json configs that are frame streams: frames per step per GPU (each step's frames are distinct and >> 126 MB L2),
# frames per in-flight chunk inside the library, description.  The driver's default is C2 (the config the metric is quoted on).
WORKLOADS = {
    "C2": dict(frames=128, slot=64, desc="C2: 1920x1080 BGR8 stream, 16 markers/frame, DICT_6X6_250, detect+pose+map update"),
    "C3": dict(frames=256, slot=128, desc="C3: 1280x720 BGR8 camera stream per GPU, 8 markers/frame, DICT_5X5_250, detect+pose+map update, merged map by NCCL all-gather"),
    "C4": dict(frames=32, slot=16, desc="C4: 3840x2160 BGR8 stream, 64 markers/frame, DICT_6X6_250, corner refine on, detect+pose+map update"),
}


def workload_cfg(name):
    w = dict(WORKLOADS[name])
    w["frames"] = int(os.environ.get("FID_BENCH_FRAMES", w["frames"]))
    w["slot"] = int(os.environ.get("FID_BENCH_SLOT", w["slot"]))
    return w


def workload_string(name):
    """config.workload -- IDENTICAL for our arm and the reference arm (the CPU arm times a bounded sample of the same stream)."""
    w = workload_cfg(name)
    nl = (w["frames"] + REALIZATIONS - 1) // REALIZATIONS
    return "%s; synthetic stream of %d frames per step per GPU = %d marker layouts x %d noise realisations (make_config_stream seed = rank)" % (w["desc"], w["frames"], nl, REALIZATIONS)


def bench_stream(name, seed):
    from fiducials_b200 import synth

    return synth.make_config_stream(name, workload_cfg(name)["frames"], seed=seed, realizations=REALIZATIONS)


def cpu_info():
    """(model name, physical cores, logical cpus) of the host the CPU arm runs on."""
    model, phys = None, set()
    try:
        for block in open("/proc/cpuinfo").read().strip().split("\n\n"):
            d = {}
            for line in block.splitlines():
                if ":" in line:
                    k, v = line.split(":", 1)
                    d[k.strip()] = v.strip()
            model = model or d.get("model name")
            if "physical id" in d and "core id" in d:
                phys.add((d["physical id"], d["core id"]))
    except OSError:
        pass
    return model or "unknown", (len(phys) or None), os.cpu_count()


def cpu_quota_cores():
    """CPU time the container may use, in cores (cgroup v2 cpu.max / v1 cfs quota); None = unlimited."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if q == "max" else float(q) / float(per)
    except Exception:
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / per
    except Exception:
        return None


def pin_to_gpu_numa_node(index):
    """Best effort: run this rank on the cores of its GPU's NUMA node (pinned staging buffers are then first-touched there)."""
    try:
        bus = subprocess.check_output(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"], text=True, timeout=20).strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read())
        if node < 0:
            return None
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def claim_stdout():
    """stdout must carry ONE JSON line: everything any library prints to fd 1 (NCCL's version banner, ...) goes to stderr instead."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def rank_info():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                      stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=2)
        except Exception:
            self.p.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback 6.65 TB/s (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# CPU reference arm (cv2): exactly the per-frame calls of the reference node
# ------------------------------------------------------------------------------------------------
_W = {}


def _cpu_worker_init(nthreads, npy_path, dict_id, K, D):
    """Worker of the throughput-mode CPU baseline (spawned, so OpenCV's thread pool is never forked)."""
    sys.path.insert(0, ROOT)
    import cv2

    cv2.setNumThreads(nthreads)
    _W["frames"] = np.load(npy_path, mmap_mode="r")
    _W["cfg"] = (dict_id, K, D)


def _cpu_worker_frame(i):
    from oracle import aruco_oracle as ao

    dict_id, K, D = _W["cfg"]
    fr = _W["frames"]
    ids, corners, rv, tv, fields = ao.detect_and_pose(np.ascontiguousarray(fr[i % len(fr)]), dict_id, K, D, FIDUCIAL_LEN)
    return len(ids)


class CpuArm:
    """The reference's CPU path on a bounded sample, in both modes (BASELINE.md section 3.5):
    reference mode  = one process, OpenCV threads = all cores (what the single-threaded node does);
    throughput mode = single-threaded worker processes, frames round-robin: one per logical core, one per
                      physical core, and -- under a cgroup CPU quota -- one and two per core of the quota (half of them on an SMT box -- the detector is memory bound and ran 30 % faster
                      that way on the 128-thread host of the B200 box).
    The worker pools are spawned once (spawn, so OpenCV's thread pool is never forked) and reused by every
    measure() call: --impl reference times K steps without paying K pool start-ups."""

    def __init__(self, frames, dict_id, K, D):
        import multiprocessing as mp
        import tempfile

        self.frames, self.dict_id, self.K, self.D = frames, dict_id, K, D
        self.ncores = os.cpu_count() or 1
        self.pools = []
        self.tmp = tempfile.NamedTemporaryFile(suffix=".npy", delete=False)
        np.save(self.tmp, np.ascontiguousarray(frames))
        self.tmp.close()
        try:
            ctx = mp.get_context("spawn")
            counts = [max(1, self.ncores)] + ([self.ncores // 2] if self.ncores >= 8 else [])
            quota = cpu_quota_cores()
            if quota and quota < self.ncores:  # a cgroup CPU quota below the CPU count: oversubscribed pools are throttled, so also
                for c in (int(round(quota)), int(round(2 * quota))):  # try one worker (and two) per core of CPU time the container owns
                    if 1 <= c < self.ncores and c not in counts:
                        counts.append(c)
            for npr in counts:
                pool = ctx.Pool(npr, initializer=_cpu_worker_init, initargs=(1, self.tmp.name, dict_id, K, D))
                pool.map(_cpu_worker_frame, range(npr), chunksize=1)  # warm-up (imports, first-call setup)
                self.pools.append((npr, pool))
        except Exception as e:  # pragma: no cover
            print("throughput-mode CPU baseline unavailable: %r" % (e,), file=sys.stderr)

    def close(self):
        for _, pool in self.pools:
            pool.terminate()
            pool.join()
        self.pools = []
        try:
            os.unlink(self.tmp.name)
        except OSError:
            pass

    def measure(self, budget_s=12.0):
        """dict(value=best fps, cores, kind, sample)."""
        import cv2

        from oracle import aruco_oracle as ao

        frames, ncores = self.frames, self.ncores

        def one(i):
            return ao.detect_and_pose(frames[i % len(frames)], self.dict_id, self.K, self.D, FIDUCIAL_LEN)

        n_modes = 1 + len(self.pools)
        # reference mode
        cv2.setNumThreads(ncores)
        one(0)
        t0 = time.perf_counter()
        n_ref = 0
        while (time.perf_counter() - t0 < budget_s / n_modes and n_ref < 4 * len(frames)) or n_ref < 3:
            one(n_ref)
            n_ref += 1
        fps_ref = n_ref / (time.perf_counter() - t0)
        # throughput mode
        fps_thr, n_thr, nproc, tried = 0.0, 0, max(1, ncores), []
        for npr, pool in self.pools:
            try:
                t0 = time.perf_counter()
                pool.map(_cpu_worker_frame, range(npr), chunksize=1)
                per_round = time.perf_counter() - t0
                rounds = int(max(1, min(8, (budget_s / n_modes) / max(per_round, 1e-3))))
                n = npr * rounds
                t0 = time.perf_counter()
                pool.map(_cpu_worker_frame, range(n), chunksize=1)
                fps = n / (time.perf_counter() - t0)
            except Exception as e:  # pragma: no cover
                print("throughput-mode CPU baseline failed: %r" % (e,), file=sys.stderr)
                continue
            tried.append("%d procs %.2f fps" % (npr, fps))
            if fps > fps_thr:
                fps_thr, n_thr, nproc = fps, n, npr
        best = max(fps_ref, fps_thr)
        model, phys, logical = cpu_info()
        return {
            "value": best,
            "unit": "frames/s",
            "cores": ncores if fps_ref >= fps_thr else nproc,
            "kind": "reference",
            "cpu_model": model,
            "physical_cores": phys,
            "logical_cpus": logical, "cgroup_cpu_quota_cores": cpu_quota_cores(),
            "sample": "cv2 %s ArucoDetector(reference params)+solvePnP+projectPoints on %d frames of the %s stream (one per marker layout: frames [::%d] of rank 0's step): "
                      "reference mode (1 proc, %d OpenCV threads) %d frames %.2f fps; throughput mode (%d procs x 1 thread) %d frames %.2f fps [%s]; value = best of all; "
                      "host: %s, %s physical cores, %d logical cpus"
                      % (cv2.__version__, len(frames), WORKLOAD, REALIZATIONS, ncores, n_ref, fps_ref, nproc, n_thr, fps_thr, ", ".join(tried), model, phys, logical or 0),
        }


def cpu_reference_fps(frames, dict_id, K, D, budget_s=12.0):
    arm = CpuArm(frames, dict_id, K, D)
    try:
        return arm.measure(budget_s)
    finally:
        arm.close()


def run_reference_arm(args):
    rank, local_rank, world = rank_info()
    if rank != 0:
        return  # rank 0 alone runs and prints the CPU arm
    if WORKLOAD == "C5":
        return run_c5(args, reference=True)
    frames, truths, K, D, dict_id = bench_stream(WORKLOAD, seed=0)  # rank 0's stream of our arm
    frames = np.ascontiguousarray(frames[::REALIZATIONS])            # bounded sample: one frame per marker layout
    per_step = []
    detail = None
    budget = max(4.0, min(20.0, 150.0 / max(1, args.steps + args.warmup)))  # whole run: a few minutes
    arm = CpuArm(frames, dict_id, K, D)
    try:
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            detail = arm.measure(budget_s=budget)
            if i >= args.warmup:
                per_step.append((detail["value"], time.perf_counter() - t0))
    finally:
        arm.close()
    fps = float(np.median([p[0] for p in per_step]))
    ms = float(np.mean([p[1] for p in per_step]) * 1e3)
    detail["value"] = fps
    out = {
        "impl": "reference",
        "metric": METRIC[WORKLOAD],
        "value": fps,
        "unit": "frames/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": ms,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": DTYPE,
        "data": "synthetic",
        "config": {"workload": workload_string(WORKLOAD)},
        "cpu_baseline": detail,
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(out)


DTYPE = "u8/i32 (threshold, contours), f32/f64 (sub-pixel, pose, map)"
METRIC = {"C2": "frames/sec 1920x1080 (detect+pose)", "C3": "frames/sec 1280x720 per-GPU camera streams (detect+pose)", "C4": "frames/sec 3840x2160 (detect+pose)",
          "C5": "map updates/sec (500 fiducials, 10k observations)"}


def parity_gate(frames, idx, out, dict_id, K, D, maxm):
    """Oracle check of frames of the BENCHED batch (BASELINE.md section 4: a parity gate beside every number).
    Same bars as tests/test_gpu_parity.py: ids identical and in identical order, corners / tvec / quaternion <= 1e-3."""
    from oracle import aruco_oracle as ao

    counts, ids, corners, tfs = out
    worst_c, worst_t, n_markers = 0.0, 0.0, 0
    for i in idx:
        ids_o, corners_o, rv, tv, fields = ao.detect_and_pose(np.ascontiguousarray(frames[i]), dict_id, K, D, FIDUCIAL_LEN)
        n = int(counts[i])
        if ids[i, :n].tolist() != ids_o.tolist():
            raise SystemExit("bench.py parity gate FAILED on frame %d: ids %s vs oracle %s" % (i, ids[i, :n].tolist(), ids_o.tolist()))
        if n == 0:
            continue
        dc = float(np.abs(corners[i, :n].reshape(n, 4, 2) - corners_o).max())
        worst_c = max(worst_c, dc)
        for m in range(n):
            t = tfs[i * maxm + m]
            worst_t = max(worst_t, float(np.abs(np.array(t.translation[:]) - fields[m]["translation"]).max()), float(np.abs(np.array(t.rotation[:]) - fields[m]["rotation"]).max()))
        n_markers += n
        if dc > 1e-3 or worst_t > 1e-3:
            raise SystemExit("bench.py parity gate FAILED on frame %d: corner diff %.3g px, pose diff %.3g" % (i, dc, worst_t))
    return {"parity_checked_frames": len(idx), "parity_checked_markers": n_markers, "max_corner_diff_px": worst_c, "max_pose_diff": worst_t,
            "bars": "ids identical and in identical order; corners, tvec, quaternion <= 1e-3 vs oracle/aruco_oracle.py (cv2) on frames of the timed batch"}


def map_rows(entries):
    """fid_map_entry list -> float64 rows: fiducial_id, num_obs, x, y, z, rx, ry, rz, variance."""
    return np.array([[e.fiducial_id, e.num_obs, e.x, e.y, e.z, e.rx, e.ry, e.rz, e.variance] for e in entries], np.float64).reshape(-1, 9)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: one DIR/<name>.npy per array, so that two builds can be compared output for output on identical inputs."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


def detection_arrays(out, maxm):
    """The results of one batch as a caller of the detect/pose path receives them, without the unused slots past each frame's
    count: markers in frame order, then in the order the library reports them."""
    from fiducials_b200.node import FiducialSlam

    counts, ids, corners, tfs = out
    nf = len(counts)
    valid = np.arange(maxm)[None, :] < counts[:, None]
    tf = np.frombuffer(bytes(tfs), FiducialSlam.TRANSFORM_DTYPE).reshape(nf, maxm)[valid]
    return {"counts": counts, "ids": ids[valid], "corners": corners.reshape(nf, maxm, 4, 2)[valid], "translation": tf["translation"], "rotation": tf["rotation"],
            "rvec": tf["rvec"], "image_error": tf["image_error"], "object_error": tf["object_error"], "fiducial_area": tf["fiducial_area"]}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_gpu_arm(args):
    import torch

    rank, local_rank, world = rank_info()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    if WORKLOAD == "C5":
        return run_c5(args, reference=False)
    torch.cuda.set_device(local_rank)
    numa_node = pin_to_gpu_numa_node(local_rank)  # before the pinned staging buffer is allocated (first touch)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # "NCCL version ..." goes to stdout, which must hold the one JSON line only
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from fiducials_b200 import _lib, synth
    from fiducials_b200.multigpu import MapExchange
    from fiducials_b200.node import MAXM, Detector, FiducialSlam, default_params

    lib = _lib.load()
    wl = workload_cfg(WORKLOAD)
    W, H, n_markers, dict_id = synth.CONFIGS[WORKLOAD]
    nf, slot_frames = wl["frames"], wl["slot"]
    frames, truths, K, D, _ = bench_stream(WORKLOAD, seed=rank)
    det = Detector(default_params(dictionary=dict_id), local_rank, W, H, slot_frames)
    slam = FiducialSlam(device=local_rank, max_fiducials=512, n_instances=1)
    exchange = MapExchange(slam, dist, torch.device("cuda", local_rank))  # merged map: stream-ordered export -> all-gather -> merge
    ident = [0, 0, 0, 0, 0, 0, 1]

    # pinned host copy + device-resident copy of the stream
    hptr = C.c_void_p()
    _lib.check(lib.fid_host_alloc(frames.nbytes, C.byref(hptr)))
    pinned = np.ctypeslib.as_array(C.cast(hptr, C.POINTER(C.c_uint8)), shape=(frames.nbytes,)).reshape(frames.shape)
    pinned[...] = frames
    dptr = C.c_void_p()
    _lib.check(lib.fid_device_alloc(det.h, frames.nbytes, C.byref(dptr)))
    _lib.check(lib.fid_memcpy_h2d(det.h, dptr, hptr, frames.nbytes))

    launches = [0]

    def submit(on_device):
        # one batch (= one step's frames) into the library's queue; returns at once
        if on_device:
            det.submit_batch(dptr.value, K, D, FIDUCIAL_LEN, on_device=True, n_frames=nf, width=W, height=H)
        else:
            det.submit_batch(pinned, K, D, FIDUCIAL_LEN)  # H2D of this batch is queued here, inside the timed region

    outs = [None] * 4

    def finish(k):
        # results of the oldest batch in flight (host arrays) + its map update.  fiducial_slam: the frames of this step are
        # one camera stream -> one message per frame; the sequential fold is enqueued asynchronously on the map's stream,
        # followed (same stream, no host synchronisation) by the export of the local map, ONE NCCL all-gather of the
        # fixed-size tables and the deterministic merge into the merged view.  The timed region ends with slam.sync().
        outs[k & 3] = det.collect_batch(outs[k & 3])
        counts, ids, corners, tfs = outs[k & 3]
        launches[0] += det.last_counters()["kernel_launches"]
        slam.update_frames(counts, tfs, ident, ident, asynchronous=True)
        launches[0] += 1
        launches[0] += exchange.step()
        return counts

    def run_steps(on_device, steps):
        # software pipeline over steps: batch k+1 is submitted before batch k is collected, so the latency-bound tail of
        # one batch (grouping, identification, pose, D2H) runs under the threshold / border-walk stages of the next.
        # Exactly `steps` batches are submitted AND collected in here.
        total = 0
        ahead = min(DEPTH - 1, steps)
        for _ in range(ahead):
            submit(on_device)
        for k in range(steps):
            if k + ahead < steps:
                submit(on_device)
            total += int(finish(k).sum())
        return total

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(on_device, steps):
        barrier()
        launches[0] = 0
        _lib.check(lib.fid_timer_start(det.h))
        t0 = time.perf_counter()
        total = run_steps(on_device, steps)
        slam.sync()
        ms = C.c_float(0)
        _lib.check(lib.fid_timer_stop(det.h, C.byref(ms)))
        wall = time.perf_counter() - t0
        barrier()
        t = torch.tensor([ms.value / 1e3, wall], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), total, launches[0]

    run_steps(True, max(args.warmup, 3))
    run_steps(False, 2)
    slam.sync()

    sampler = ClockSampler(local_rank)
    sampler.start()
    dev_s, dev_wall, n_markers_found, n_launch = timed(True, args.steps)
    stage_ms = det.last_stage_ms()  # stages of the last batch call (nf frames)
    counters = det.last_counters()
    last_out = outs[(args.steps - 1) & 3]
    if args.dump_outputs and rank == 0:  # before the e2e pass reuses the output buffers
        dump_outputs(args.dump_outputs, dict(detection_arrays(last_out, MAXM), map_entries=map_rows(slam.entries()), merged_map_entries=map_rows(slam.merged_entries())))
    e2e_s, e2e_wall, _, _ = timed(False, args.steps)
    clocks = sampler.stop()
    n_merged = len(slam.merged_entries())

    # parity gate on frames of the timed batch (every rank checks its own stream; a mismatch ends the run)
    n_gate = int(os.environ.get("FID_BENCH_PARITY_FRAMES", "16"))
    gate_idx = list(range(0, nf, max(1, nf // max(1, n_gate))))[:n_gate]
    parity = parity_gate(frames, gate_idx, last_out, dict_id, K, D, MAXM) if n_gate > 0 else {"parity_checked_frames": 0}

    # extra (not the metric): latency of ONE frame through the synchronous per-frame call the reference node makes
    # (imageCallback + poseEstimateCallback), host frame in, host results out, nothing else on the GPU
    single_ms = None
    if rank == 0:
        try:
            det1 = Detector(default_params(dictionary=dict_id), local_rank, W, H, 1)
            one = np.ascontiguousarray(pinned[:1])
            for _ in range(3):
                det1.detect_pose_batch(one, K, D, FIDUCIAL_LEN)
            t0 = time.perf_counter()
            for i in range(20):
                det1.detect_pose_batch(np.ascontiguousarray(pinned[i % nf : i % nf + 1]), K, D, FIDUCIAL_LEN)
            single_ms = (time.perf_counter() - t0) / 20 * 1e3
            det1.close()
        except Exception as e:  # pragma: no cover
            print("single-frame latency probe failed: %r" % (e,), file=sys.stderr)

    frames_total = nf * args.steps * world
    value = frames_total / dev_s
    e2e_value = frames_total / e2e_s

    if rank == 0:
        n_scales = 13
        peak, peak_src = measured_hbm_peak()
        bytes_per_frame = 3 * W * H + n_scales * W * H / 8.0  # SURVEY 8d: BGR in, 13 bit planes out
        # (1) the threshold stage timed ALONE on one chunk (what a launch costs; compared with the burst copy peak)
        chunk = min(slot_frames, nf)
        alone = C.c_float(0)
        _lib.check(lib.fid_debug_time_threshold(det.h, chunk, dptr, W, H, W * 3, W * 3 * H, 5, C.byref(alone)), "fid_debug_time_threshold")
        algo_bytes = bytes_per_frame * chunk
        achieved = algo_bytes / (alone.value / 1e3) / 1e9
        # (2) the same stage inside the pipelined step (CUDA events on its stream, while up to three other
        #     chunks run their own stages on the same SMs): share of the step
        n_launch_thr = (nf + slot_frames - 1) // slot_frames
        thr_pipe_ms = stage_ms["threshold"] / n_launch_thr
        total_stage = sum(v for k, v in stage_ms.items() if k not in ("h2d", "d2h") and not k.startswith("walk_r"))
        traffic, traffic_src = None, None
        try:  # DRAM bytes of the kernel from the committed ncu --set full capture of this round (per frame, scaled to this launch)
            tj = json.load(open(os.path.join(ROOT, "profiles", "r02_threshold_traffic.json")))
            if tj.get("workload") == WORKLOAD:
                traffic = float(tj["dram_bytes_per_frame"]) * chunk
                traffic_src = "profiles/r02_threshold_traffic.json (ncu --set full capture of the same kernel and workload; not re-measured by this run)"
        except Exception:
            pass
        roofline = {
            "bound": "hbm",
            "kernel": ("k_threshold_mma (BGR->gray + 13 adaptive thresholds on the int8 tensor cores + halo tiles + start cracks, one launch)" if os.environ.get("FID_THRESH") == "mma" else "k_threshold<FAST> (threshold stage in one launch: BGR->gray fused into the region load, summed-area table in shared memory, 13 thresholds, halo tiles + start cracks)"),
            "achieved": achieved,
            "peak": peak,
            "unit": "GB/s",
            "frac": achieved / peak,
            "traffic": traffic,
            "traffic_source": traffic_src,
            "peak_source": peak_src + "; kernel timed alone -> burst figure",
            "algorithmic_bytes_per_launch": algo_bytes,
            "frames_per_launch": chunk,
            "launch_ms": alone.value,
            "in_pipeline": {
                "launch_ms": thr_pipe_ms,
                "achieved": bytes_per_frame * slot_frames / (thr_pipe_ms / 1e3) / 1e9 if thr_pipe_ms > 0 else None,
                "share_of_step": stage_ms["threshold"] / total_stage if total_stage else None,
                "note": "event-bracketed on the launching stream while other chunks' kernels share the SMs",
            },
            "stage_ms_per_batch": stage_ms,
            "work_per_batch": counters,
        }
        if os.environ.get("FID_BENCH_SKIP_CPU"):  # profiling runs (ncu) only
            cpu = {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference", "sample": "skipped (FID_BENCH_SKIP_CPU set)"}
        elif world > 1:  # the CPU baseline is a rank-0, N = 1 measurement (the host cores do not multiply with the GPUs)
            cpu = {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference", "sample": "measured at N = 1 only: see the 1-GPU line / --impl reference"}
        else:
            cpu = cpu_reference_fps(np.ascontiguousarray(frames[::REALIZATIONS]), dict_id, K, D, budget_s=16.0)
        d2h = nf * (4 + MAXM * 4 + MAXM * 32 + MAXM * C.sizeof(_lib.fid_transform))
        out = {
            "metric": METRIC[WORKLOAD],
            "value": value,
            "unit": "frames/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": max(args.warmup, 3),
            "ms_per_step": dev_s * 1e3 / args.steps,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": DTYPE,
            "data": "synthetic",
            "config": {
                "workload": workload_string(WORKLOAD),
                "frames_per_step_per_gpu": nf,
                "l2": "inputs larger than L2 (%d MB of distinct frames per step vs 126 MB L2)" % (frames.nbytes // 2**20),
                "parallelism": ("one camera stream per GPU, no collective on detect/pose; per step the local map tables are exported, all-gathered (NCCL) and merged on the "
                                "map's CUDA stream without blocking the host") if world > 1 else "1 GPU",
                "markers_found_per_step": n_markers_found // max(1, args.steps),
                "merged_map_fiducials": n_merged,
                "numa_node": numa_node,
            },
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": int(frames.nbytes), "d2h_bytes_per_step": int(d2h), "ms_per_step": e2e_s * 1e3 / args.steps,
                    "h2d_gbs": frames.nbytes * args.steps / e2e_s / 1e9,
                    "note": "raw BGR8 frames over PCIe: the end-to-end figure is bounded by the pinned-copy bandwidth of the host link (h2d_gbs is what this run moved)"},
            "gpu_launches": n_launch,
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "parity": parity,
            "wallclock_s": {"device_resident": dev_wall, "e2e": e2e_wall},
            "single_frame_latency_ms": single_ms,
        }
        emit(out)
    lib.fid_device_free(det.h, dptr)
    lib.fid_host_free(hptr)
    det.close()
    slam.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def run_c5(args, reference):
    """BASELINE.json config C5: 500-fiducial / 10k-observation pose-graph sequence (synth.make_c5_sequence) through the
    fiducial_slam update.  A step = the whole 1000-message sequence into a fresh map (fiducial 0 pinned), one launch of
    fid_map_update_sequence per GPU (every rank folds its own replica: the fold is sequential per map, SURVEY 8e -- "replicas only");
    value = observations/s over all ranks.  --impl reference: the same fold compiled for the host (oracle/_ref, one core)."""
    from fiducials_b200 import synth

    rank, local_rank, world = rank_info()
    msgs, seed_entry = synth.make_c5_sequence(1000, seed=0)
    n_obs = sum(len(m) for m in msgs)
    ident7 = [0, 0, 0, 0, 0, 0, 1]
    metric = METRIC["C5"]
    workload = "C5: 500 fiducials on a 25x20 ceiling grid, 1000 messages / %d observations (synth.make_c5_sequence seed 0), fiducial 0 pinned, sequential fiducial_slam fold per map" % n_obs
    if reference:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import bench_c5

        per = []
        for i in range(args.warmup + args.steps):
            dt = bench_c5.cpu_fold_seconds(msgs, seed_entry)
            if i >= args.warmup:
                per.append(dt)
        dt = float(np.median(per))
        model, phys, logical = cpu_info()
        val = n_obs / dt
        out = {"impl": "reference", "metric": metric, "value": val, "unit": "observations/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": {"workload": workload},
               "cpu_baseline": {"value": val, "unit": "observations/s", "cores": 1, "kind": bench_c5.cpu_fold_kind()[0], "cpu_model": model, "physical_cores": phys, "logical_cpus": logical, "cgroup_cpu_quota_cores": cpu_quota_cores(),
                                "sample": "the whole sequence through " + bench_c5.cpu_fold_kind()[1] + ", one core",
                                "arithmetic_only_port": bench_c5.cpu_port_info(msgs, seed_entry)},
               "e2e": {"value": val, "unit": "observations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(out)
        return
    import torch

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from fiducials_b200 import _lib
    from fiducials_b200.node import FiducialSlam

    slam = FiducialSlam(device=local_rank, max_fiducials=512, n_instances=1)
    offsets = np.zeros((1, len(msgs) + 1), np.int32)
    flat = []
    for k, m in enumerate(msgs):
        offsets[0, k] = len(flat)
        flat.extend(m)
    offsets[0, len(msgs)] = len(flat)
    obs = np.zeros(len(flat), FiducialSlam.TRANSFORM_DTYPE)
    for i, ft in enumerate(flat):
        obs[i]["fiducial_id"] = ft["fiducial_id"]
        obs[i]["translation"] = ft["translation"]
        obs[i]["rotation"] = ft["rotation"]
        obs[i]["image_error"], obs[i]["object_error"], obs[i]["fiducial_area"] = ft["image_error"], ft["object_error"], ft["fiducial_area"]

    def one():
        slam.clear(0)
        slam.loadMap([seed_entry])
        t0 = time.perf_counter()
        slam.replay_raw(offsets, obs, ident7, ident7)  # H2D of the observations + the fold + sync
        return time.perf_counter() - t0

    for _ in range(max(args.warmup, 3)):
        one()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    per = [one() for _ in range(args.steps)]
    dt = float(np.mean(per))
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t[0])
    ents = slam.entries(0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"map_entries": map_rows(ents)})
    # the north-star's batched SE(3) Gauss-Newton over the same observations (fid_map_refine; new, parity unpinned): cost, the
    # reference's plane-fit metric (fiducial_slam/scripts/fit_plane.py; the synthetic ceiling is the plane z = 2.5) and wall time
    refine = None
    if rank == 0:
        from oracle import refine_oracle as ro

        pts0 = [[e.x, e.y, e.z] for e in ents]
        truth = np.array([[float(e.fiducial_id % 25), float(e.fiducial_id // 25), 2.5] for e in ents])
        t0 = time.perf_counter()
        st = slam.refine(msgs)
        refine_s = time.perf_counter() - t0
        ents_r = slam.entries(0)
        pts1 = [[e.x, e.y, e.z] for e in ents_r]
        refine = {"seconds": refine_s, "solve_kernel_ms": st.solve_ms, "seconds_note": "seconds = the Python call (message marshalling + edge build on the host + solve); solve_kernel_ms = the one cooperative kernel, CUDA events", "edges": st.n_edges, "free_poses": st.n_free, "gauss_newton_steps": st.iterations, "kernel_launches": st.kernel_launches,
                  "cost_initial": st.initial_cost, "cost_final": st.final_cost,
                  "plane_fit_residual_before": ro.plane_fit_residual(pts0), "plane_fit_residual_after": ro.plane_fit_residual(pts1),
                  "max_position_error_before_m": float(np.abs(np.array(pts0) - truth).max()), "max_position_error_after_m": float(np.abs(np.array(pts1) - truth).max()),
                  "rms_position_error_before_m": float(np.sqrt(np.mean((np.array(pts0) - truth) ** 2))), "rms_position_error_after_m": float(np.sqrt(np.mean((np.array(pts1) - truth) ** 2)))}
    # parity gate: the numpy restatement over a 250-message prefix is covered by tests/test_gpu_slam.py::test_c5_pose_graph_sequence;
    # here: the host-compiled fold of the FULL sequence must agree with the device's map to 1e-8
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import bench_c5

    ref_entries = bench_c5.cpu_fold_entries(msgs, seed_entry)
    worst = 0.0
    assert [e.fiducial_id for e in ents] == [r[0] for r in ref_entries], "C5 parity gate: fiducial sets differ"
    for e, r in zip(ents, ref_entries):
        worst = max(worst, max(abs(e.x - r[1]), abs(e.y - r[2]), abs(e.z - r[3]), abs(e.rx - r[4]), abs(e.ry - r[5]), abs(e.rz - r[6])))
    if worst > 1e-8:
        raise SystemExit("C5 parity gate FAILED: %.3g" % worst)
    if rank == 0:
        val = n_obs * world / dt
        cpu_dt = bench_c5.cpu_fold_seconds(msgs, seed_entry)
        model, phys, logical = cpu_info()
        out = {"metric": metric, "value": val, "unit": "observations/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dt * 1e3,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
               "config": {"workload": workload, "parallelism": "replicas only: every rank folds its own copy of the sequence (the fold is sequential per map)", "map_fiducials": len(ents)},
               "e2e": {"value": val, "unit": "observations/s", "h2d_bytes_per_step": int(obs.nbytes + offsets.nbytes), "d2h_bytes_per_step": 0, "note": "value already includes the H2D of the observations"},
               "gpu_launches": args.steps, "parity": {"max_entry_diff_vs_host_fold": worst, "entries": len(ents)}, "batch_gauss_newton_refine": refine,
               "cpu_baseline": {"value": n_obs / cpu_dt, "unit": "observations/s", "cores": 1, "kind": bench_c5.cpu_fold_kind()[0], "cpu_model": model, "physical_cores": phys, "logical_cpus": logical, "cgroup_cpu_quota_cores": cpu_quota_cores(),
                                "sample": "the whole sequence through " + bench_c5.cpu_fold_kind()[1] + ", one core, %.2f ms" % (cpu_dt * 1e3),
                                "arithmetic_only_port": bench_c5.cpu_port_info(msgs, seed_entry)},
               "roofline": {"bound": "latency", "note": "sequential scalar-variance fold (SURVEY 8d): no roofline fraction is meaningful; report observations/s and ms per sequence"}}
        emit(out)
    slam.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2", choices=["C2", "C3", "C4", "C5"], help="BASELINE.json config (the driver's default, C2, is the one the metric is quoted on)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy (float32/float64; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    global WORKLOAD
    WORKLOAD = args.workload
    claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
