#!/usr/bin/env python
"""bench.py -- frames/s of MaskFusion::processFrame on a synthetic 640x480 .klg replay.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A step is one processFrame call (one pass of the per-frame dense hot path) on one frame of a seeded synthetic replay.

N = 1  workload = BASELINE.json configs[1]: "-static" single-model path, 640x480, the background store pre-populated to ~4.7M
       surfels (capacity 2176^2, the reference's rounding of 5M, Model.cpp:101-106).
  value : frames/s with every frame already resident in HBM when the timed region starts
  e2e   : frames/s through the reference-facing C-ABI call mf_process_frame with pinned HOST buffers (H2D copies of rgb+depth and
          the D2H pose read-back inside the timed region)
  roofline     : dominant kernel (largest share of device time, measured live with CUDA events on the launching stream) as
                 algorithmic GB/s against MEASURED_PEAKS.json
  cpu_baseline : the CPU oracle (oracle/, a restatement of the reference; the reference's own GL/CUDA program cannot run here)
                 on a bounded sample of the same workload
  legs next to the main line (never instead of it): cpu_seg (configs[0]: the CPU part of MfSegmentation on 1 core / all cores),
  ref_cuda (the reference's own CUDA kernels recompiled, one model-frame of tracking in its calling pattern), multi_object
  (configs[2]: 3 tracked objects + the Mask R-CNN backbone on the same GPU), eight_objects (configs[3] on one GPU), ate (ATE-RMSE of
  every model's exported trajectory against the oracle on the first frames of the 8-object replay), backbone.

N > 1  (torchrun) workload = configs[3]: ONE 640x480 replay with 8 tracked objects, the object Models sharded over the N GPUs
       (strong scaling: the replay is the same for every N).  The three exchanges of a frame -- frame-packet broadcast, pose-row
       all-gather, 64-bit MIN all-reduce of the ID-projection keys -- are NCCL calls issued inside the library on its stream.
  value : frames/s, inputs resident in rank 0's HBM; e2e: the same with pinned host inputs on rank 0 and the pose read back
  single_process_same_workload : the same replay through one context on rank 0's GPU (the baseline the sharding is measured against)
  replicas : secondary leg, N independent configs[1] replays (the -static path has one model and does not shard)

--dump-outputs DIR (N = 1): after the timed passes, what the last processFrame call left for its caller is written as DIR/<name>.npy
(float32 / float64, ~40 MB): the background pose and pose log, the surfel count and a fixed seeded sample of the surfel store's rows,
and the predicted view.  The replay and the pre-populated store are seeded, so two builds run with the same arguments can be
compared output for output.

Nothing is written into the tree (it may be read-only): no bytecode caches, the replay file goes to the temporary directory.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

W, H = 640, 480
CAPACITY = 2176 * 2176            # 64*floor(sqrt(5e6)/64) squared, Model.cpp:101-106
PREPOP = 4_300_000                # dense room surfels uploaded after frame 0 (+ ~0.3M from the frame itself)
DUMP_ROWS = 1 << 19               # surfel rows kept by --dump-outputs (24 MB of the ~230 MB store)
METRIC = "frames/sec on 640x480 .klg replay"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle reasons sampled through NVML (the same counters nvidia-smi prints) every ~2 ms
    during the timed regions; the timed region of this workload is too short for `nvidia-smi -lms`."""

    def __init__(self, gpu):
        self.gpu, self.sm, self.reasons, self.stop_flag, self.ok = gpu, [], 0, False, False
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = gpu
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                idx = int(vis.split(",")[gpu])
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:          # noqa: BLE001
            self.err = str(e)

    def start(self):
        # rank 0 samples its GPU; the other ranks do not poll NVML (eight processes polling the driver every 2 ms next to ~30 launches per
        # millisecond each were a suspect for the replica leg's efficiency loss at N = 4 / 8 in round 1)
        if not self.ok or int(os.environ.get("RANK", "0")) != 0:
            self.ok = self.ok and int(os.environ.get("RANK", "0")) == 0
            return
        self.stop_flag = False
        self.t = threading.Thread(target=self._loop, daemon=True); self.t.start()

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.reasons |= nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:           # noqa: BLE001
                pass
            time.sleep(0.004)

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self.stop_flag = True
        self.t.join(timeout=1)
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        reasons = [k for k, bit in names.items() if self.reasons & bit]
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": float(self.max), "reasons": reasons, "samples": len(self.sm)}


def make_replay(n_frames, seed):
    """synthetic replay written to a raw .klg and read back through KlgLogReader (the loader is outside the timed region)"""
    import maskfusion_b200 as mfb
    from maskfusion_b200.synth import SynthScene
    n_frames = min(n_frames, 96)           # unique frames; longer runs replay them forwards/backwards (camera reverses)
    sc = SynthScene(W, H, n_objects=0, seed=seed)
    d16 = np.zeros((n_frames + 1, H, W), np.uint16); rgb = np.zeros((n_frames + 1, H, W, 3), np.uint8)
    for t in range(n_frames):
        r, _, _, _, d = sc.render(t)
        rgb[t], d16[t] = r, d
    fd, path = tempfile.mkstemp(prefix="mfb200_bench_", suffix=".klg")
    os.close(fd)
    mfb.write_klg(path, np.arange(n_frames + 1, dtype=np.int64) * 33333, d16, rgb)     # +1: hasMore() never yields the last frame (N11)
    rd = mfb.KlgLogReader(path, W, H)
    frames = []
    while rd.hasMore():
        frames.append(rd.getNext())
    rd.close()
    os.remove(path)
    return sc, frames


def prepopulate(mf, sc):
    """fill the background store to ~4.7M surfels: dense synthetic room cloud in the model frame (= camera-0 frame)"""
    from maskfusion_b200.synth import dense_room_surfels
    gm = mf.getBackgroundModel()
    cur = gm.downloadMap()
    room = dense_room_surfels(sc, PREPOP, time=1, conf=20.0)
    Tinv = np.linalg.inv(sc.camera_pose(0))
    room[:, 0:3] = (room[:, 0:3].astype(np.float64) @ Tinv[:3, :3].T + Tinv[:3, 3]).astype(np.float32)
    room[:, 8:11] = (room[:, 8:11].astype(np.float64) @ Tinv[:3, :3].T).astype(np.float32)
    allv = np.concatenate([cur, room], 0)
    gm.uploadMap(allv)
    return allv.shape[0]


# algorithmic bytes of one launch, S = live surfels, P = pixels (DESIGN.md "kernels and rooflines")
def algorithmic_bytes(name, S, P):
    table = {
        "k_index_project": 32 * S,                   # position + colour/time planes (normal plane never read)
        "k_index_resolve": 8 * P + 52 * P,
        "k_clean_p1": 32 * S + 1 * (S + P),       # position + colour/time planes, keep flag (round 2: the index projection rides in the same stream)
        "k_clean_p2": 48 * P + 4 * P,              # ~one candidate per pixel neighbourhood; window reads hit L2 (the candidate list is ~S/3 long: see DESIGN.md)
        "k_clean_scatter": 48 * S + 48 * S + 1 * (S + P),       # ping-pong copy of the whole store (MFB200_CLEAN_INPLACE=0)
        "k_clean_compact": 1 * (S + P),                      # in-place compaction: keep flags; the moved tail (96 B per surfel behind the first removal) is data dependent
        "k_splat_project": 16 * S,                   # position plane for every surfel; +32 B only for in-frustum stable ones
        "k_splat_resolve": 8 * P + 38 * P + 36 * P,
        "k_associate": 13 * P + 93 * P,
        "k_bilateral": 8 * P,
        "k_track_persistent": (552 + 713) * P,       # SURVEY 8(d): ICP 48 B x P_l and photometric 62 B x P_l per iteration over the 10/5/4 schedule
    }
    return table.get(name)


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel`, from the newest committed `ncu --set full`
    summary under profiles/ (scripts/summarize_ncu.py); None when no capture of that kernel is committed"""
    import glob
    import re
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", f"*_prof_{kernel}.txt")))
    if not files:
        return None, None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    tot = 0.0
    for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
        m = re.search(re.escape(key) + r" = ([0-9.]+) (\w+)", open(files[-1]).read())
        if not m:
            return None, None
        tot += float(m.group(1)) * unit.get(m.group(2), 1.0)
    return int(tot), os.path.basename(files[-1])


def dump_outputs(mf, out_dir):
    """what the last processFrame call left for its caller: pose, pose log, the surfel store (DUMP_ROWS rows at seeded positions when it
    holds more) and the predicted view (splat image, vertex, normal, time)"""
    gm = mf.getBackgroundModel()
    surfels = gm.downloadMap()
    if len(surfels) > DUMP_ROWS:
        surfels = surfels[np.sort(np.random.default_rng(0).choice(len(surfels), DUMP_ROWS, replace=False))]
    image, vertex, normal, stamp = gm.prediction()
    arrays = {"pose": gm.getPose(), "pose_log": gm.poseLog(), "surfel_count": np.array([gm.lastCount()], np.float64), "surfels": surfels,
              "prediction_image": image.astype(np.float32), "prediction_vertex": vertex, "prediction_normal": normal,
              "prediction_time": stamp.astype(np.float32)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def static_leg(torch, mfb, stream, local, rank, world, K, Wm, dump_dir=None):
    """configs[1]: the main line at N = 1, the `replicas` leg at N > 1"""
    n_need = 1 + 3 * (Wm + K) + 2
    sc, frames = make_replay(n_need, seed=rank)
    nu = len(frames)

    def fidx(j):                        # ping-pong over the unique frames: 0..nu-1, nu-2..1, 0..
        period = 2 * (nu - 1)
        r = j % period
        return r if r < nu else period - r
    cfg = mfb.default_config(W, H, capacityGlobal=CAPACITY)        # GUI defaults: ICP+RGB (w=20), SO3, -static
    mf = mfb.MaskFusion(cfg, device=local, stream=stream.cuda_stream)
    rgb0, d0, ts0 = frames[0]
    mf.processFrame(rgb0, d0, ts0)
    prepopulate(mf, sc)
    # pinned host staging (e2e) and device-resident copies (value)
    host_rgb = [torch.from_numpy(f[0]).pin_memory() for f in frames]
    host_d = [torch.from_numpy(f[1]).pin_memory() for f in frames]
    dev_rgb = [t.cuda() for t in host_rgb]
    dev_d = [t.cuda() for t in host_d]
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(first, on_device):
        for i in range(Wm):
            j = fidx(first + i)
            mf.processFramePtr((dev_rgb if on_device else host_rgb)[j].data_ptr(), (dev_d if on_device else host_d)[j].data_ptr(), (first + i) * 33333, on_device)
        mf.sync()
        barrier()
        l0 = mf.kernelLaunches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(K):
            j = fidx(first + Wm + i)
            mf.processFramePtr((dev_rgb if on_device else host_rgb)[j].data_ptr(), (dev_d if on_device else host_d)[j].data_ptr(), (first + Wm + i) * 33333, on_device)
            if not on_device:
                mf.getBackgroundModel().getPose()              # the step's result, read on the host every frame
        e1.record(stream)
        mf.sync()
        barrier()
        return e0.elapsed_time(e1), mf.kernelLaunches() - l0

    sampler = ClockSampler(local); sampler.start()
    dev_runs = [timed(1, True)]
    ms_e2e, _ = timed(1 + Wm + K, False)                   # e2e: pinned host buffers through the C ABI
    dev_runs.append(timed(1, True))                        # the device-resident region twice more: the spread of the timed region is reported
    dev_runs.append(timed(1, True))
    clocks = sampler.stop()
    mf.setProfiling(True)                                  # same region again with the in-stream CUDA-event stage timer
    ms_prof, _ = timed(1 + 2 * (Wm + K), True)
    stages = mf.stageTimes()
    mf.setProfiling(False)
    S_live = mf.getBackgroundModel().lastCount()
    if dump_dir:
        dump_outputs(mf, dump_dir)
    ms_all = sorted(r[0] for r in dev_runs)
    ms_dev, launches = ms_all[1], dev_runs[0][1]           # median of three passes
    if world > 1:
        t = torch.tensor([ms_dev, ms_e2e], device="cuda", dtype=torch.float64)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms_dev, ms_e2e = float(t[0]), float(t[1])
    mf.close()
    return {"ms_dev": ms_dev, "ms_e2e": ms_e2e, "ms_prof": ms_prof, "ms_passes": ms_all, "launches": launches, "clocks": clocks, "stages": stages, "S_live": S_live}


def roofline_of(stages, S_live, K, Wm, ms_prof):
    P = W * H
    kern = {k: v for k, v in stages.items() if k.startswith("k_")}
    # the tracking schedule of a frame is one logical kernel in two launches (cluster kernel: SO3 + level 2, persistent kernel: levels 1-0);
    # its algorithmic bytes (SURVEY 8d: 1265 B per pixel over the whole schedule) are divided by the time of both
    two_launches = "k_track_cluster" in kern and "k_track_persistent" in kern          # MFB200_TRACK_CLUSTER=1 (default: one launch)
    if two_launches:
        a, b = kern.pop("k_track_cluster"), kern.pop("k_track_persistent")
        kern["k_track_persistent"] = (b[0], a[1] + b[1])
    total_ms = sum(v[1] for v in stages.values())
    dom = max(kern, key=lambda k: kern[k][1])
    peak, peak_src = load_peaks()
    ab = algorithmic_bytes(dom, S_live, P)
    avg_ms = kern[dom][1] / kern[dom][0]
    achieved = (ab / 1e9) / (avg_ms / 1e3) if ab else None
    shares = {k: round(v[1] / total_ms, 4) for k, v in sorted(stages.items(), key=lambda kv: -kv[1][1])[:14]}
    traffic, traffic_src = ncu_traffic(dom)
    per_kernel = {}
    for k, (n, ms) in kern.items():
        b = algorithmic_bytes(k, S_live, P)
        if b and n:
            g = (b / 1e9) / (ms / n / 1e3)
            per_kernel[k] = {"launches_per_step": round(n / (K + Wm), 2), "avg_ms": round(ms / n, 5), "GBps": round(g, 1), "frac": round(g / peak, 4)}
    return {"kernel": dom if not (two_launches and dom == "k_track_persistent") else "k_track_cluster + k_track_persistent (one tracking schedule, two launches)", "bound": "hbm", "achieved": round(achieved, 1) if achieved else None, "peak": peak, "peak_source": peak_src,
            "unit": "GB/s", "frac": round(achieved / peak, 4) if achieved else None, "traffic": traffic,
            "traffic_source": traffic_src, "avg_launch_ms": round(avg_ms, 5), "algorithmic_bytes_per_launch": ab,
            "note": "the tracking kernels walk 29 dependent Gauss-Newton reductions over maps that stay in L2 (DRAM traffic << algorithmic bytes): "
                    "bound by that serial chain, not by HBM; the streaming surfel passes are listed in `kernels`",
            "time_shares": shares, "kernels": per_kernel, "profiled_ms_per_step": round(ms_prof / K, 4)}


# ------------------------------------------------------------------------------------------------------------------------------
# multi-object replays (configs[2] / configs[3]): SURVEY 8(d) table scene, masks as inputs (the reference's -maskdir mode)
# ------------------------------------------------------------------------------------------------------------------------------
MULTI_KW = dict(capacityGlobal=1000000, capacityObject=262144, enableMultipleModels=1, icpWeight=20.0, so3=1, trackAllModels=1, modelSpawnOffset=3)


def multi_frames(n_objects, n_frames):
    from maskfusion_b200.synth import render_sequence, SynthScene
    fr = render_sequence(range(n_frames), width=W, height=H, n_objects=n_objects, seed=0, layout="table")
    sc = SynthScene(W, H, n_objects=n_objects, seed=0, layout="table")
    cls = np.array([0] + [o.class_id for o in sc.objects], np.int32)
    return [(f[0], f[1], f[2]) for f in fr], cls


def single_process_multi(torch, mfb, stream, local, frames, cls, timed_from, backbone_every=0, want_poses=False):
    """one context, all models on this GPU; frames [timed_from, end) timed twice: device-resident inputs, then pinned host inputs + pose
    read-back per frame.  backbone_every = k > 0: the ResNet-101-FPN backbone runs on a second stream every k-th frame (configs[2])"""
    cfg = mfb.default_config(W, H, **MULTI_KW)
    mf = mfb.MaskFusion(cfg, device=local, stream=stream.cuda_stream)
    n = len(frames)
    host = [(torch.from_numpy(f[0]).pin_memory(), torch.from_numpy(f[1]).pin_memory(), torch.from_numpy(np.ascontiguousarray(f[2])).pin_memory()) for f in frames]
    dev = [(a.cuda(), b.cuda(), c.cuda()) for a, b, c in host]
    bb = None
    if backbone_every:
        bstream = torch.cuda.Stream()
        bb = mfb.Backbone(1024, seed=1, stream=bstream.cuda_stream)
        mf.attachBackbone(bb, backbone_every)
    torch.cuda.synchronize()
    mf.setFrameClasses(cls)

    def run(lo, hi, on_device, read_pose):
        src = dev if on_device else host
        for t in range(lo, hi):
            mf.processFramePtr(src[t][0].data_ptr(), src[t][1].data_ptr(), t * 33333, on_device, mask_ptr=src[t][2].data_ptr())
            if read_pose:
                mf.getBackgroundModel().getPose()
    run(0, timed_from, True, False)
    mf.sync(); torch.cuda.synchronize()
    l0 = mf.kernelLaunches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    run(timed_from, n, True, False)
    e1.record(stream)
    mf.sync(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    launches = mf.kernelLaunches() - l0
    models = mf.getModels()
    res = {"value": round((n - timed_from) / (ms / 1e3), 2), "unit": "frames/s", "ms_per_step": round(ms / (n - timed_from), 4), "frames": n - timed_from,
           "models": len(models), "surfels": [m.lastCount() for m in models], "gpu_launches": int(launches)}
    if want_poses:
        res["_poselogs"] = [m.poseLog() for m in models]
    mf.close()
    if bb is not None:
        bb.close()
    return res


def oracle_multi_poselogs(frames, cls, n):
    """the CPU oracle on the first n frames of a multi-object replay -> per-model pose logs (test infrastructure: the ATE checker)"""
    import ctypes as C
    from tests import oracle_lib as ol
    orc = ol.OraclePipeline(ol.default_config(W, H, **MULTI_KW))
    L = orc.L
    L.orc_mf_process_frame_ex.argtypes = [C.c_void_p] * 3 + [C.c_int64, C.c_void_p, C.c_void_p, C.c_int]
    t0 = time.time()
    for t in range(n):
        rgb, depth, mask = frames[t]
        L.orc_mf_process_frame_ex(orc.h, ol.ptr(np.ascontiguousarray(rgb)), ol.ptr(np.ascontiguousarray(depth)), t * 33333, ol.ptr(np.ascontiguousarray(mask)),
                                  ol.ptr(cls), len(cls))
    dt = time.time() - t0
    logs = []
    i = 0
    while True:
        try:
            m = orc.model(i)
        except Exception:          # noqa: BLE001
            break
        if i >= 64 or m.nlog <= 0 or not m.log:
            break
        logs.append(np.array([m.log[k] for k in range(m.nlog * 8)]).reshape(-1, 8))
        i += 1
        if i >= _oracle_nmodels(orc):
            break
    return logs, dt


def _oracle_nmodels(orc):
    import ctypes as C
    from tests.test_gpu_multi import MFS
    return int(C.cast(orc.h, C.POINTER(MFS)).contents.nmodels)


def ate_rmse(lo, lc):
    to = {int(r[0]): r[1:4] for r in lo}; tc = {int(r[0]): r[1:4] for r in lc}
    common = sorted(set(to) & set(tc))
    if not common:
        return None
    d = np.array([to[k] - tc[k] for k in common])
    return float(np.sqrt(np.mean(np.sum(d * d, axis=1))))


def cpu_seg_baseline():
    """BASELINE configs[0] / SURVEY 8(d)(i): the CPU part of MfSegmentation::performSegmentation (MfSegmentation.cpp:208-538, restated in
    oracle/orc_mfseg.c, its OpenCV pieces pinned against cv2) on ONE 640x480 frame of the 3-object scene: one core (the reference is
    single-threaded there) and all host cores with a straightforward OpenMP split"""
    from tests import oracle_lib as ol
    fr = ol.segmentation_frame()
    cores = min(os.cpu_count() or 1, 32)
    _, ncomp, _, t1 = ol.run_mfseg_cpu(fr, threads=1, repeats=15)
    _, _, _, tn = ol.run_mfseg_cpu(fr, threads=cores, repeats=15)
    return {"workload": "configs[0]: single 640x480 RGB-D frame, CPU geometric-segmentation tail (connected components, edge removal, overlap voting)",
            "one_core_ms": round(t1 * 1e3, 3), "all_cores_ms": round(tn * 1e3, 3), "cores": cores, "components": ncomp, "kind": "port",
            "frames_per_s_one_core": round(1.0 / t1, 1), "frames_per_s_all_cores": round(1.0 / tn, 1)}


def run_ours(args, rank, world):
    import torch
    import maskfusion_b200 as mfb
    local = int(os.environ.get("LOCAL_RANK", 0))
    pre = None
    if world > 1 and rank == 0:
        # the loader rank renders the replay before CUDA / NCCL exist in this process (the renderer forks worker processes)
        n_pre = min(34 + args.warmup + args.steps, 160)
        pre = multi_frames(8, n_pre)
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(minutes=20))
    K, Wm = args.steps, args.warmup
    stream = torch.cuda.Stream()          # explicit: the default stream's NULL handle would make mf_create open a private stream the events cannot see
    torch.cuda.set_stream(stream)
    if world > 1:
        return run_sharded(args, rank, world, torch, mfb, stream, local, pre)
    st = static_leg(torch, mfb, stream, local, rank, world, K, Wm, dump_dir=args.dump_outputs)
    P = W * H
    fps = K / (st["ms_dev"] / 1e3)
    fps_e2e = K / (st["ms_e2e"] / 1e3)
    out = {
        "metric": METRIC, "value": round(fps, 3), "unit": "frames/s", "n_gpus": 1, "steps": K, "warmup": Wm,
        "ms_per_step": round(st["ms_dev"] / K, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: -static single model, 640x480 synthetic .klg replay, ICP+RGB+SO3 tracking + surfel fuse, 1 B200",
                   "surfels_live": int(st["S_live"]), "surfel_capacity": CAPACITY, "tracking": "GUI defaults icpWeight=20 so3=1 pyramid=1",
                   "l2": "surfel store (227 MB: three float4 planes x 4.73 M capacity, one copy) + per-frame maps exceed the 126 MB L2 between steps (no explicit flush)",
                   "parallelism": "single", "numerics": "fp32 per element; Gauss-Newton sums in fp64 of exact products, rounded to the reference's float record"},
        "timed_region": {"passes_ms": [round(m, 3) for m in st["ms_passes"]], "value_from": "median of three device-resident passes",
                         "min_ms_per_step": round(st["ms_passes"][0] / K, 4), "max_ms_per_step": round(st["ms_passes"][-1] / K, 4)},
        "e2e": {"value": round(fps_e2e, 3), "unit": "frames/s", "h2d_bytes_per_step": P * 3 + P * 4, "d2h_bytes_per_step": 160 + 64},
        "gpu_launches": int(st["launches"]),
        "clocks": st["clocks"],
        "roofline": roofline_of(st["stages"], st["S_live"], K, Wm, st["ms_prof"]),
    }
    if os.environ.get("MFB200_BENCH_LEGS", "1") == "0":          # A/B runs of the main line only
        print(json.dumps(out))
        return
    out["cpu_baseline"] = cpu_baseline(sample_frames=4)

    def leg(name, fn):
        try:
            out[name] = fn()
        except Exception as e:          # noqa: BLE001  (the main line must survive a failure of an optional leg)
            out[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
    leg("cpu_seg", cpu_seg_baseline)

    def ref_cuda():
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import time_ref_track
        r = time_ref_track.run(10)
        trk = sum(v[1] for k, v in st["stages"].items() if k.startswith("k_track")) / max(1, st["stages"].get("k_track_persistent", (1, 0))[0])
        r["this_library_tracking_us_per_model_frame"] = round(trk * 1e3, 1)
        return r
    leg("ref_cuda", ref_cuda)
    n8 = 72
    frames8 = cls8 = None

    def eight():
        nonlocal frames8, cls8
        frames8, cls8 = multi_frames(8, n8)
        r = single_process_multi(torch, mfb, stream, local, frames8, cls8, timed_from=34, want_poses=True)
        r["workload"] = "configs[3] on ONE GPU: 8 tracked objects (17-23 k pixels each, table scene of SURVEY 8d) + background, 640x480, masks as inputs"
        return r
    leg("eight_objects", eight)

    def ate():
        logs_c = out["eight_objects"].pop("_poselogs")
        n_ate = 40
        logs_o, dt = oracle_multi_poselogs(frames8, cls8, n_ate)
        vals = [ate_rmse(lo, lc) for lo, lc in zip(logs_o, logs_c)]
        return {"unit": "m", "frames": n_ate, "models": len(vals), "background_ate_rmse": vals[0], "worst_object_ate_rmse": max(vals[1:]) if len(vals) > 1 else None,
                "per_model": vals, "bit_identical_poses": bool(all(v == 0.0 for v in vals)),
                "against": f"CPU oracle (restatement of the reference) on the first {n_ate} frames of the 8-object replay ({dt:.0f} s on {os.environ.get('OMP_NUM_THREADS')} threads); "
                           "exported trajectories as MaskFusion.cpp:577-592 logs them, no alignment"}
    leg("ate", ate)
    if isinstance(out.get("eight_objects"), dict):
        out["eight_objects"].pop("_poselogs", None)

    def configs4():
        # BASELINE configs[4] on ONE GPU: 1280x720, 16 objects (table scene, three rows), capacities 50M global / 1M per object as the
        # reference rounds them (Model.cpp:101-106: 7040^2 and 960^2), the background store pre-populated to ~30M live surfels
        from maskfusion_b200.synth import render_sequence, SynthScene, dense_room_surfels
        W4, H4, n4, t0 = 1280, 720, 48, 36
        kw = dict(width=W4, height=H4, n_objects=16, seed=0, layout="table")
        fr = render_sequence(range(n4), **kw)
        sc = SynthScene(W4, H4, n_objects=16, seed=0, layout="table")
        cls = np.array([0] + [o.class_id for o in sc.objects], np.int32)
        cfg = mfb.default_config(W4, H4, capacityGlobal=7040 * 7040, capacityObject=960 * 960, enableMultipleModels=1, icpWeight=20.0, so3=1, trackAllModels=1,
                                 modelSpawnOffset=1, fx=792.0, fy=792.0, cx=640.0, cy=360.0)
        mf = mfb.MaskFusion(cfg, device=local, stream=stream.cuda_stream)
        dev = [(torch.from_numpy(f[0]).cuda(), torch.from_numpy(f[1]).cuda(), torch.from_numpy(np.ascontiguousarray(f[2])).cuda()) for f in fr]
        mf.setFrameClasses(cls)

        def run(lo, hi):
            for t in range(lo, hi):
                mf.processFramePtr(dev[t][0].data_ptr(), dev[t][1].data_ptr(), t * 33333, True, mask_ptr=dev[t][2].data_ptr())
        run(0, 1)
        gm = mf.getBackgroundModel()
        cur = gm.downloadMap()
        room = dense_room_surfels(sc, 30_000_000, time=1, conf=20.0)
        Tinv = np.linalg.inv(sc.camera_pose(0))
        room[:, 0:3] = (room[:, 0:3].astype(np.float64) @ Tinv[:3, :3].T + Tinv[:3, 3]).astype(np.float32)
        room[:, 8:11] = (room[:, 8:11].astype(np.float64) @ Tinv[:3, :3].T).astype(np.float32)
        gm.uploadMap(np.concatenate([cur, room], 0))
        del room
        run(1, t0)
        mf.sync(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        run(t0, n4)
        e1.record(stream)
        mf.sync(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        models = mf.getModels()
        r = {"value": round((n4 - t0) / (ms / 1e3), 2), "unit": "frames/s", "ms_per_step": round(ms / (n4 - t0), 3), "frames": n4 - t0, "models": len(models),
             "surfels": [m.lastCount() for m in models], "surfel_capacity": [7040 * 7040, 960 * 960],
             "hbm_store_bytes": int(48 * (7040 * 7040 + (len(models) - 1) * 960 * 960)),
             "workload": "configs[4] on ONE GPU: 1280x720, 16 objects (table scene) + background, 50M global / 1M per-object capacities, background pre-populated "
                         "to ~30M live surfels, masks as inputs; inputs resident in HBM"}
        mf.close()
        return r
    if os.environ.get("MFB200_BENCH_CONFIGS4", "1") != "0":
        leg("configs4_720p_16_objects", configs4)

    def three():
        fr3, cls3 = multi_frames(3, 60)
        r = single_process_multi(torch, mfb, stream, local, fr3, cls3, timed_from=20)
        try:
            rb = single_process_multi(torch, mfb, stream, local, fr3, cls3, timed_from=20, backbone_every=5)
            r["with_backbone_every_5th_frame"] = {"value": rb["value"], "ms_per_step": rb["ms_per_step"],
                                                  "note": "ResNet-101-FPN forward (1024x1024, synthetic weights) enqueued on a second stream every 5th frame (the reference's sidecar runs at ~5 Hz)"}
        except Exception as e:          # noqa: BLE001
            r["with_backbone_every_5th_frame"] = {"error": f"{type(e).__name__}: {e}"[:300]}
        r["workload"] = "configs[2]: 3 tracked objects, 640x480, 1 B200, Mask R-CNN backbone on the same GPU; masks are inputs (-maskdir mode: the R-CNN heads are not built)"
        return r
    leg("multi_object", three)

    def backbone():
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import bench_cnn
        return bench_cnn.run(1024, iters=5, warm=2)
    leg("backbone", backbone)
    print(json.dumps(out))


def run_sharded(args, rank, world, torch, mfb, stream, local, pre):
    """N > 1: configs[3], object Models sharded over the ranks (in-library NCCL exchange); replicas of configs[1] as the secondary leg"""
    import torch.distributed as dist
    from maskfusion_b200.sharding import ShardedMaskFusion
    K, Wm = args.steps, args.warmup
    warm_to = 34                                            # 8 objects spawned (one every 3 frames), 30 static frames over
    n = min(warm_to + Wm + K, 160)
    K = n - warm_to - Wm
    frames = cls = None
    single = None
    if rank == 0:
        frames, cls = pre
        frames = frames[:n]
        single = single_process_multi(torch, mfb, stream, local, frames, cls, timed_from=warm_to + Wm)
    dist.barrier()
    cfg = mfb.default_config(W, H, **MULTI_KW)
    smf = ShardedMaskFusion(cfg, device=local)
    clsp = None
    if rank == 0:
        host = [(torch.from_numpy(f[0]).pin_memory(), torch.from_numpy(f[1]).pin_memory(), torch.from_numpy(np.ascontiguousarray(f[2])).pin_memory()) for f in frames]
        dev = [(a.cuda(), b.cuda(), c.cuda()) for a, b, c in host]
        clsp = np.ascontiguousarray(cls, np.int32)
    torch.cuda.synchronize()

    def step(t, on_device, read_pose=False):
        if rank == 0:
            src = dev if on_device else host
            smf.processFramePtr(src[t][0].data_ptr(), src[t][1].data_ptr(), t * 33333, src[t][2].data_ptr(), clsp.ctypes.data, len(clsp), on_device)
        else:
            smf.processFramePtr(0, 0, 0, 0, 0, 0, False)
        if read_pose:
            smf.mf.getBackgroundModel().getPose()

    def timed(lo, hi, on_device, read_pose):
        smf.mf.sync(); dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(smf.stream)
        for t in range(lo, hi):
            step(t, on_device, read_pose)
        e1.record(smf.stream)
        smf.mf.sync(); dist.barrier(); torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms[0])
    sampler = ClockSampler(local); sampler.start()
    for t in range(warm_to + Wm):
        step(t, True)
    s0 = smf.stats()
    l0 = smf.mf.kernelLaunches()
    ms_dev = timed(warm_to + Wm, n, True, False)
    launches = smf.mf.kernelLaunches() - l0
    s1 = smf.stats()
    clocks = sampler.stop()
    # e2e: the same frames again are not available (the replay has moved on): time the NEXT K frames with host inputs would need more
    # frames; instead a second sharded context replays the whole sequence with pinned host inputs and a pose read-back per frame
    models = smf.models()
    owners = [smf.owner(i) for i in range(len(models))]
    smf.close()
    smf2 = ShardedMaskFusion(cfg, device=local)
    smf_keep = smf
    smf = smf2
    for t in range(warm_to + Wm):
        step(t, False)
    ms_e2e = timed(warm_to + Wm, n, False, True)
    smf.close()
    del smf_keep
    # secondary leg: replicas of configs[1]
    try:
        if os.environ.get("MFB200_BENCH_LEGS", "1") == "0":
            raise RuntimeError("skipped (MFB200_BENCH_LEGS=0)")
        st = static_leg(torch, mfb, stream, local, rank, world, min(args.steps, 60), args.warmup)
        kk = min(args.steps, 60)
        replicas = {"value": round(world * kk / (st["ms_dev"] / 1e3), 2), "unit": "frames/s", "ms_per_step": round(st["ms_dev"] / kk, 4),
                    "e2e": round(world * kk / (st["ms_e2e"] / 1e3), 2),
                    "workload": "configs[1] -static, one independent replay per GPU (no collective on the data path), total frames/s"}
    except Exception as e:          # noqa: BLE001
        replicas = {"error": f"{type(e).__name__}: {e}"[:300]}
    if rank == 0:
        P = W * H
        per_frame = (s1["bytes"] - s0["bytes"]) / K
        out = {
            "metric": METRIC, "value": round(K / (ms_dev / 1e3), 3), "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": round(ms_dev / K, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[3]: 8 tracked objects, 640x480 synthetic replay (table scene, SURVEY 8d), object Models sharded across the GPUs, "
                                   "NCCL RGB-D broadcast + pose gather + ID-key MIN all-reduce issued inside the library",
                       "parallelism": "object-sharded", "models": len(models), "owners": owners, "tracking": "ICP+RGB (w=20) + SO3, every model tracked",
                       "l2": "per-rank working set (frame maps + stores of the local models) fits L2; every frame is new input", "masks": "inputs (-maskdir mode)"},
            "e2e": {"value": round(K / (ms_e2e / 1e3), 3), "unit": "frames/s", "h2d_bytes_per_step": P * 8 + 1040, "d2h_bytes_per_step": 8464},
            "gpu_launches": int(launches), "clocks": clocks,
            "collectives": {"transport": s1["transport"], "comm_nranks_seen": s1["nranks"], "nccl_version": s1["nccl_version"],
                            "calls_per_frame": round((s1["calls"] - s0["calls"]) / K, 2), "bytes_per_frame": int(per_frame),
                            "what": "ncclBroadcast frame packet (2.46 MB) + ncclAllGather pose rows (8 KB per rank) + ncclAllReduce(min, u64) projection keys (2.46 MB)"},
            "single_process_same_workload": single,
            "speedup_vs_single_process": round((K / (ms_dev / 1e3)) / single["value"], 3) if single else None,
            "replicas": replicas,
        }
        print(json.dumps(out))
    dist.barrier()
    dist.destroy_process_group()


def cpu_baseline(sample_frames):
    """CPU oracle on a bounded sample of the same workload (same surfel count, same defaults)"""
    from tests import oracle_lib as ol
    from maskfusion_b200.synth import dense_room_surfels, SynthScene
    import ctypes as C
    sc = SynthScene(W, H, n_objects=0, seed=0)
    threads = int(os.environ.get("OMP_NUM_THREADS", os.cpu_count() or 1))
    p = ol.OraclePipeline(ol.default_config(W, H, capacityGlobal=CAPACITY))
    rgb, depth, *_ = sc.render(0)
    p.process_frame(rgb, depth, 0)
    m = p.L.orc_mf_model(p.h, 0)
    cur = p.surfels(0).copy()
    room = dense_room_surfels(sc, PREPOP, time=1, conf=20.0)
    Tinv = np.linalg.inv(sc.camera_pose(0))
    room[:, 0:3] = (room[:, 0:3].astype(np.float64) @ Tinv[:3, :3].T + Tinv[:3, 3]).astype(np.float32)
    room[:, 8:11] = (room[:, 8:11].astype(np.float64) @ Tinv[:3, :3].T).astype(np.float32)
    allv = np.ascontiguousarray(np.concatenate([cur, room], 0))
    C.memmove(m.contents.surf[m.contents.target], allv.ctypes.data, allv.nbytes)
    m.contents.count = allv.shape[0]
    fr = [sc.render(t)[:2] for t in range(1, 1 + sample_frames)]
    t0 = time.time()
    for i, (r, d) in enumerate(fr):
        p.process_frame(r, d, (i + 1) * 33333)
    dt = time.time() - t0
    return {"value": round(sample_frames / dt, 4), "unit": "frames/s", "cores": threads, "kind": "port",
            "sample": f"{sample_frames} frames of the same replay, {allv.shape[0]} surfels; OpenMP in every per-pixel / per-surfel pass (sums and ordered compaction keep the sequential order, results bit-identical to one thread)"}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU restatement (oracle port) on the host cores; rank 0 only"""
    if rank != 0:
        return
    K = max(1, min(args.steps, 6))
    cb = cpu_baseline(sample_frames=K)
    out = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": 0,
           "ms_per_step": round(1e3 / cb["value"], 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic",
           "config": {"workload": "configs[1]: -static single model, 640x480 synthetic replay, same surfel count and defaults as the CUDA arm",
                      "note": "the reference's own CUDA+OpenGL program cannot run in this environment (no OpenGL/Pangolin/Eigen/OpenCV); this arm is the CPU oracle port"},
           "cpu_baseline": cb,
           "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (N = 1)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (world > 1 or args.impl != "ours"):
        ap.error("--dump-outputs applies to the single-GPU run of this library")
    if args.impl == "reference":
        # the CPU arm uses all host threads it can, also under torchrun (which exports OMP_NUM_THREADS=1 for its workers)
        os.environ["OMP_NUM_THREADS"] = str(min(os.cpu_count() or 1, 32))
    else:
        os.environ.setdefault("OMP_NUM_THREADS", str(min(os.cpu_count() or 1, 32)))  # oracle's OpenMP sections (cpu_baseline)
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world)


if __name__ == "__main__":
    main()
