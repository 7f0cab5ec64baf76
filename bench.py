#!/usr/bin/env python
"""bench.py -- headline benchmark of cudasift_b200 (BASELINE.json metric, config #2).

  python bench.py --gpus N --steps K --warmup W            # the product (default N=1)
  python bench.py --impl reference --gpus N ...            # the unmodified reference build
  (N>1: launched by `python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N`)

A "step" is `rounds` passes of ExtractSift over a batch of synthetic 1920x1080 float images that are resident in HBM
(32 distinct device buffers = 265 MB > the 126 MB L2, so every pass re-reads its inputs from DRAM).  `rounds` is chosen
by the same rule in both arms so that the K timed steps cover >= 7680 images per GPU: the timed region then lasts
>= 0.3 s and the in-process NVML sampler sees it (--steps 20 -> 12 rounds = 384 images per step; --steps 300 -> 1).
Product arm:
  value    images/s, device-resident inputs, through the BATCHED extractor API (one launch per stage for a whole
           batch; every image has its own record slot, counts come back to the host every step)
  e2e      the same metric with HOST (pinned) buffers: H2D of every image and D2H of every result inside the timed
           region, through cs_extractor_submit_host_batch / cs_extractor_wait_batch
  dropin   the reference's own call -- mangled ExtractSift(SiftData&, CudaImage&, ...) on a device-resident
           CudaImage, synchronous, with and without the host copy of the records
  roofline per-stage times of one batch (CUDA events on the extractor's stream), HBM roofline of the pyramid kernel
           and of the detector, packed-FP32 roofline of the detector
  match    MatchSiftData 2000 x 2000 and 10000 x 10000 (BASELINE config #3), exact and tensor-core paths
  allpairs (N > 1) BASELINE config #5: per-GPU ExtractSift + ONE NCCL all-gather + all-pairs match
  cpu_baseline (N = 1) the oracle port on the host cores + OpenCV SIFT
  --dump-outputs DIR  writes the keypoints of the last timed step as .npy files (dump_outputs), so that two builds can be
           compared output for output on the same seeded inputs
Reference arm (--impl reference): the unmodified reference library (oracle/_ref/libcudasift_ref.so) through its own
C++ API in a process that never loads libcudasift_b200.so: same images, same config, same statistics.
One JSON line on stdout (rank 0).
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W, H, OCTAVES, INIT_BLUR, THRESH, MAX_PTS = 1920, 1080, 5, 1.0, 3.0, 32768
REC = 576
# packed FP32 instructions (FFMA2 + FADD2 + FMUL2, warp level) the detector executes per 1080p image, and the DRAM
# traffic of the dominant kernels per image: one ncu --set full capture of a batch of 16 (profiles/r02_prof_extract.txt,
# profiles/r02_sass_hist_detect3.txt): (48.23 + 33.16 + 12.06) M / 16, (178.7 + 5.3) MB / 16, (152.3 + 116.9) MB / 16
DETECT_PACKED_WARP_INSTR = 5.84e6
DETECT_DRAM_BYTES = 11.5e6
PYR_DRAM_BYTES = 16.8e6
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libcudasift_ref.so")


def level_sizes(w=W, h=H, n=OCTAVES):
    out = []
    for _ in range(n):
        out.append((w, h))
        w, h = w // 2, h // 2
    return out


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)", d
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)", {}


MIN_TIMED_IMAGES = 7680   # per GPU: the timed region lasts >= 0.3 s at 24k images/s, so that clocks can be sampled in it


def rounds_per_step(args):
    """A step = `rounds` passes over the `batch` device-resident images.  Chosen by the same rule in both arms so that
    K steps cover at least MIN_TIMED_IMAGES images per GPU (the driver runs --steps 20: 12 rounds of 32 images)."""
    if args.rounds > 0:
        return args.rounds
    return max(1, -(-MIN_TIMED_IMAGES // (max(1, args.steps) * args.batch)))


def workload_config(batch, distinct, pitch, features, rounds=1):
    """The `config` object: identical in both arms (same inputs, same parameters, same statistic)."""
    return {"workload": "ExtractSift 1920x1080 float, 5 octaves, initBlur 1.0, thresh 3.0 (BASELINE config #2)",
            "images_per_step_per_gpu": batch * rounds, "distinct_images": distinct,
            "l2_policy": "inputs larger than L2 (%d device images = %.0f MB per GPU, %d pass(es) over them per step)"
                         % (batch, batch * pitch * H * 4 / 1e6, rounds),
            "features_per_image": round(float(features), 1),
            "parallelism": "images sharded one process per GPU, no collective"}


# ------------------------------------------------------------------------------------------ host placement
def bind_numa(gpu_index):
    """Pin this process to the CPUs of the GPU's NUMA node BEFORE any pinned allocation: at 8 GPUs the host->device
    path is 8 x 50 GB/s of pinned reads, which only works if every rank reads its own socket's memory."""
    info = {"bound": False}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:          # nvml gives an 8-digit domain, sysfs uses 4
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return info
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            info = {"bound": True, "numa_node": node, "cpus": len(cpus)}
    except Exception as e:           # no NVML / sysfs: run unbound and say so
        info["error"] = str(e)[:80]
    return info


class ClockSampler:
    """SM clock, power and throttle reasons sampled in-process through NVML every 20 ms during the timed region."""

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = False
        self.h = None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        except Exception:
            self.h = None

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        if self.h is None:
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"], "samples": 0}
        self.stop_flag = True
        self.t.join(timeout=1)
        nv = self.nv
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = None
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80}
        reasons = set()
        for _, _, rs in self.samples:
            for k, bit in names.items():
                if rs & bit:
                    reasons.add(k)
        sm = [s[0] for s in self.samples]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": round(max([s[1] for s in self.samples]), 1) if sm else None}


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def init_dist(world, local):
    if world <= 1:
        return None
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return dist


def reduce_max(dist, x):
    if dist is None:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def synth_module(standalone=False):
    """Synthetic inputs.  The reference arm loads synth.py as a plain module: it never imports the cudasift_b200 package."""
    if not standalone:
        from cudasift_b200 import synth
        return synth
    d = os.path.join(ROOT, "cudasift_b200")
    if d not in sys.path:
        sys.path.append(d)
    import synth
    return synth


def make_images(rank, distinct, standalone=False):
    synth_image = synth_module(standalone).synth_image
    return [synth_image(W, H, seed=1000 + 100 * rank + i) for i in range(distinct)]


# ------------------------------------------------------------------------------------------ product arm
def run_product(args):
    rank, world, local = dist_env()
    numa = bind_numa(local)
    import cudasift_b200 as cs
    cs.InitCuda(local)
    dist = init_dist(world, local)
    L = cs.lib()

    def sync_all():
        L.cs_device_sync()
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    B, S = args.batch, args.streams
    b = B // S
    assert b * S == B and 1 <= b <= L.cs_max_batch(), "batch must be streams x (1..%d)" % L.cs_max_batch()
    pitch = cs.iAlignUp(W, 128)
    imgs = make_images(rank, args.distinct)
    dbufs = []
    for i in range(B):                                # B distinct device buffers (> L2)
        img = cs.CudaImage().Allocate(W, H, pitch, False, None, imgs[i % len(imgs)])
        img.Download()
        dbufs.append(img)
    ptrs = [d.d_data for d in dbufs]
    exs = [cs.Extractor(W, H, OCTAVES, MAX_PTS, False, batch=b) for _ in range(S)]
    ev0 = [L.cs_event_create() for _ in range(S)]
    ev1 = [L.cs_event_create() for _ in range(S)]

    R = rounds_per_step(args)

    def step_device():
        for _ in range(R):
            for s in range(S):
                exs[s].submit_device_batch(ptrs[s * b:(s + 1) * b], pitch, INIT_BLUR, THRESH, 0.0)

    for _ in range(args.warmup):
        step_device()
    [ex.wait_batch(b) for ex in exs]
    # --- timed region 1: device-resident inputs ---
    sampler = ClockSampler(local)
    sync_all()
    sampler.start()
    launches0 = L.cs_launch_count()
    for s in range(S):
        L.cs_event_record(ev0[s], exs[s].handle)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_device()
    for s in range(S):
        L.cs_event_record(ev1[s], exs[s].handle)
    counts = []
    for ex in exs:
        counts += ex.wait_batch(b)
    sync_all()
    wall = time.perf_counter() - t0
    dev_ms = max(L.cs_event_elapsed_ms(ev0[0], ev1[s]) for s in range(S))
    launches = L.cs_launch_count() - launches0
    clocks = sampler.stop()
    dev_ms = reduce_max(dist, dev_ms)
    wall = reduce_max(dist, wall)
    n_images = args.steps * B * R * world
    value = n_images / (dev_ms / 1e3)
    pts_per_image = float(np.mean(counts))            # all B images of the last step
    if args.dump_outputs and rank == 0:               # outside the timed region, before anything reuses the record slots
        dump_outputs(args.dump_outputs, [exs[s].device_points_at(i, counts[s * b + i]) for s in range(S) for i in range(b)])

    # --- timed region 2: end to end through the C ABI with host (pinned) buffers ---
    hptrs = []
    for s in range(S):
        for i in range(b):
            hp = L.cs_extractor_host_image_at(exs[s].handle, i)
            ctypes.memmove(hp, imgs[(s * b + i) % len(imgs)].ctypes.data, W * H * 4)
            hptrs.append(hp)
    e2e_rounds = max(16, min(args.steps, 200) // 12)  # batches per extractor: >= 512 images (~80 ms at the PCIe rate)

    def run_e2e(rounds):
        d2h = 0
        busy = [False] * S
        for _ in range(rounds):
            for s in range(S):
                if busy[s]:
                    d2h += sum(exs[s].wait_batch(b)) * REC + 16 * b
                exs[s].submit_host_batch(hptrs[s * b:(s + 1) * b], INIT_BLUR, THRESH, 0.0)
                busy[s] = True
        for s in range(S):
            if busy[s]:
                d2h += sum(exs[s].wait_batch(b)) * REC + 16 * b
        return d2h

    run_e2e(1)
    sync_all()
    t0 = time.perf_counter()
    d2h_bytes = run_e2e(e2e_rounds)
    sync_all()
    e2e_s = reduce_max(dist, time.perf_counter() - t0)
    e2e_images = e2e_rounds * B
    e2e_value = e2e_images * world / e2e_s
    h2d_gbs = e2e_images * W * H * 4 / e2e_s / 1e9

    out = {
        "metric": "1920x1080 images/sec ExtractSift", "value": round(value, 1), "unit": "images/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dev_ms / args.steps, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(B, len(imgs), pitch, pts_per_image, R),
        "api": "cs_extractor_submit_device_batch: %d extractor(s) x batch %d, one launch per stage per batch, CUDA graph, "
               "own record slot per image, counts read back every step" % (S, b),
        "clocks": clocks, "numa": numa,
        "e2e": {"value": round(e2e_value, 1), "unit": "images/s", "h2d_bytes_per_step": B * R * W * H * 4,
                "d2h_bytes_per_step": int(d2h_bytes / e2e_images * B * R), "images": e2e_images * world,
                "h2d_gbs_per_rank": round(h2d_gbs, 1),
                "api": "cs_extractor_submit_host_batch / cs_extractor_wait_batch (pinned host buffers, %d batches of %d in flight)" % (S, b)},
        "gpu_launches": int(launches * world),
        "wall_s": round(wall, 4),
    }
    if rank == 0:
        out["dropin"] = bench_dropin(cs, imgs, pitch)
        out["roofline"] = bench_roofline(cs, exs[0], ptrs[:b], pitch, b, value, world, pts_per_image)
        out["match"] = bench_match(cs)
    if world > 1:
        ap = bench_allpairs(cs, dist, rank, world)
        if rank == 0:
            out["allpairs"] = ap
    if rank == 0:
        if world == 1 and not args.no_cpu:
            out["cpu_baseline"] = cpu_baseline(imgs)
        print(json.dumps(out), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


DUMP_FIELDS = ("xpos", "ypos", "scale", "sharpness", "edgeness", "orientation", "subsampling")
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, per_image):
    """What ExtractSift hands its caller for each image of the last timed step, as float arrays:
    counts.npy (float64, keypoints per image), keypoints.npy (float32, one row of DUMP_FIELDS per keypoint) and
    descriptors.npy (float32, 128 per keypoint); images in order, each image's keypoints in canonical order (the device
    appends them in no fixed order).  The match fields of the records are not written: extraction leaves them unset.
    Above DUMP_MAX_BYTES in all, a fixed seeded sample of keypoint rows is written, and rows.npy (float64) names them."""
    os.makedirs(out_dir, exist_ok=True)
    recs = np.concatenate([p[np.lexsort((p["orientation"], p["scale"], p["xpos"], p["ypos"], p["subsampling"]))]
                           for p in per_image])
    out = {"counts": np.array([len(p) for p in per_image], np.float64),
           "keypoints": np.stack([recs[f] for f in DUMP_FIELDS], axis=1).astype(np.float32),
           "descriptors": np.ascontiguousarray(recs["data"], np.float32)}
    row_bytes = 4 * (len(DUMP_FIELDS) + 128)
    room = DUMP_MAX_BYTES - out["counts"].nbytes - 4 * 128           # 128: the header of each .npy file
    if len(recs) * row_bytes > room:
        rows = np.sort(np.random.default_rng(0).choice(len(recs), room // (row_bytes + 8), replace=False))
        out.update(keypoints=out["keypoints"][rows], descriptors=out["descriptors"][rows], rows=rows.astype(np.float64))
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def bench_dropin(cs, imgs, pitch, n=48):
    """The reference-shaped call: mangled ExtractSift on a device-resident CudaImage, synchronous."""
    import reflib
    from cudasift_b200 import build
    lib = reflib.CxxSiftLib(build.LIB)
    c = ctypes
    images = [lib.image(imgs[i % len(imgs)]) for i in range(8)]
    tmp = lib._alloc(W, H, OCTAVES, False)
    res = {}
    for name, host in (("with_host_copy", True), ("device_only", False)):
        sd = reflib.CSiftData()
        lib._init(c.byref(sd), MAX_PTS, host, True)
        for i in range(4):
            lib._extract(c.byref(sd), c.byref(images[i % 8]), OCTAVES, INIT_BLUR, THRESH, 0.0, False, tmp)
        t0 = time.perf_counter()
        for i in range(n):
            lib._extract(c.byref(sd), c.byref(images[i % 8]), OCTAVES, INIT_BLUR, THRESH, 0.0, False, tmp)
        dt = time.perf_counter() - t0
        res[name] = {"images_per_s": round(n / dt, 1), "ms_per_call": round(dt / n * 1e3, 4), "numPts": sd.numPts}
        lib._freedata(c.byref(sd))
    lib._free(tmp)
    res["api"] = "ExtractSift(SiftData&, CudaImage&, 5, 1.0, 3.0, 0, false, tempMemory): device-resident image, one call at a time"
    return res


def bench_roofline(cs, ex, ptrs, pitch, b, value, world, pts_per_image):
    prof = []
    for i in range(8):
        n, ms = ex.profile_batch(ptrs, pitch, INIT_BLUR, THRESH, 0.0)
        prof.append(ms)
    pa_ms, chain_ms, detect_ms, describe_ms, total_ms = (np.array(prof[2:]).mean(axis=0) / b)
    lv = level_sizes()
    detect_bytes = sum(4 * w * h for w, h in lv)                       # each octave base image read once
    pyr_bytes = 2 * 4 * W * H + 4 * lv[1][0] * lv[1][1]                # read input, write level 0, write level 1
    pipeline_bytes = 4 * W * H + sum(2 * 4 * w * h for w, h in lv) + REC * pts_per_image   # SURVEY 8(d)
    peak, how, pk = peaks()
    ach = detect_bytes / (detect_ms * 1e-3) / 1e9
    sm_mhz = float(pk.get("sm_max_mhz", 1965.0))
    fp32_floor_ms = DETECT_PACKED_WARP_INSTR * 2 / (4 * 148) / (sm_mhz * 1e6) * 1e3      # 2 cycles per packed op and SMSP
    pyr_gbs = pyr_bytes / (pa_ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": "detect3_kernel (8-scale blur + DoG + 3x3x3 extrema, all octaves, whole batch per launch)",
            "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
            "traffic": DETECT_DRAM_BYTES * b, "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full "
            "capture of detect3_kernel (profiles/r02_prof_extract.txt), per launch of a batch of %d" % b,
            "peak_source": how, "algorithmic_bytes_per_launch": detect_bytes * b, "units_per_launch": b,
            "avg_launch_ms": round(float(detect_ms * b), 4),
            "stage_ms": {"lowpass_scaledown": round(float(pa_ms), 4), "scaledown_chain": round(float(chain_ms), 4),
                         "detect": round(float(detect_ms), 4), "describe": round(float(describe_ms), 4),
                         "pipeline_total": round(float(total_ms), 4), "note": "per image = per-launch time / %d images" % b},
            "detect_fp32_pipe": {"packed_warp_instr_per_image": DETECT_PACKED_WARP_INSTR, "floor_ms": round(fp32_floor_ms, 4),
                                 "frac": round(fp32_floor_ms / float(detect_ms), 4),
                                 "note": "the detector is FP32-bound, not HBM-bound: ~127 FP32 operations per pixel that parity "
                                         "fixes, against 4 bytes; floor = packed instructions x 2 cycles / (4 SMSP x 148 SM)"},
            "pyramid": {"kernel": "pyr_lowpass_sd_kernel (LowPass + first ScaleDown, TMA-fed)", "bound": "hbm",
                        "algorithmic_bytes_per_image": pyr_bytes, "achieved": round(pyr_gbs, 1), "peak": peak,
                        "frac": round(pyr_gbs / peak, 4), "traffic": PYR_DRAM_BYTES * b,
                        "traffic_source": "ncu capture, profiles/r02_prof_extract.txt"},
            "pipeline_algorithmic_bytes": int(pipeline_bytes),
            "pipeline_frac_at_value": round(pipeline_bytes * value / world / 1e9 / peak, 4)}


def bench_match(cs):
    """BASELINE.json config #3: MatchSiftData 2000 x 2000 then 10000 x 10000 synthetic 128-D descriptors."""
    from cudasift_b200.synth import synth_descriptors
    _, _, pk = peaks()
    tpeak = float(pk.get("bf16_tflops", 0.0)) or 1693.0
    res = {}
    for n in (2000, 10000):
        s1, s2 = synth_descriptors(n, 1), synth_descriptors(n, 2)
        d1 = cs.InitSiftData(cs.SiftData(), n, False, True)
        d2 = cs.InitSiftData(cs.SiftData(), n, False, True)
        d1._buf.upload(s1); d2._buf.upload(s2)
        d1.numPts = d2.numPts = n
        r = {}
        for mode, name in ((1, "exact_fp32"), (2, "tensor")):
            for _ in range(3):
                cs.MatchSiftData(d1, d2, mode=mode)
            ts = [cs.MatchSiftData(d1, d2, mode=mode) for _ in range(30)]
            ms = float(np.median(ts))
            r[name] = {"ms": round(ms, 4), "gpair_per_s": round(n * n / (ms * 1e-3) / 1e9, 2),
                       "tflops_algorithmic": round(2 * n * n * 128 / (ms * 1e-3) / 1e12, 2)}
        r["stats_tensor"] = cs.match_stats()
        t = r["tensor"]
        # three FP16 MMAs (hi*hi + hi*lo + lo*hi) per algorithmic product
        r["tensor_roofline"] = {"bound": "tensor", "kernel": "t3_gemm_kernel (tcgen05.mma kind::f16, M128 N128 K16, A in TMEM, K_eff = 384)",
                                "achieved_algorithmic": t["tflops_algorithmic"], "achieved_executed": round(3 * t["tflops_algorithmic"], 2),
                                "peak": tpeak, "unit": "TFLOP/s", "frac_algorithmic": round(t["tflops_algorithmic"] / tpeak, 4),
                                "frac_executed": round(3 * t["tflops_algorithmic"] / tpeak, 4),
                                "peak_source": "MEASURED_PEAKS.json bf16_tflops (cuBLAS burst)" if pk else "fallback",
                                "note": "whole MatchSiftData call (prep + GEMM + resolve + D2H of the 5 result fields)"}
        res["n%d" % n] = r
        cs.FreeSiftData(d1); cs.FreeSiftData(d2)
    return res


def bench_allpairs(cs, dist, rank, world, cap=4096, reps=5):
    """BASELINE config #5: every rank extracts ONE image, one all_gather_into_tensor moves the SiftPoint arrays
    (fixed capacity, the count rides in a header record: no second collective), rank g then matches its set against
    every other.  Timed with CUDA events; verified against the oracle on rank 0 outside the timed region."""
    import torch
    from cudasift_b200.synth import synth_image
    L = cs.lib()
    img = synth_image(W, H, seed=5000 + rank)
    d_img = torch.from_numpy(np.ascontiguousarray(img)).cuda()          # pitch == width (1920 % 128 == 0)
    send = torch.zeros((cap + 1) * REC, dtype=torch.uint8, device="cuda")   # record 0 = header, records 1.. = points
    recv = torch.empty(world * (cap + 1) * REC, dtype=torch.uint8, device="cuda")
    pts_ptr = send.data_ptr() + REC
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    t_ext, t_ag, t_match = [], [], []
    counts = None
    for rep in range(reps + 1):
        torch.cuda.synchronize()
        dist.barrier()
        e[0].record()
        n = L.cs_extract(d_img.data_ptr(), W, H, W, OCTAVES, INIT_BLUR, THRESH, 0.0, 0, None, pts_ptr, None, cap)
        assert 0 < n <= cap, L.cs_last_error()
        send[:4] = torch.tensor([n], dtype=torch.int32).view(torch.uint8).cuda(non_blocking=True)
        e[1].record()
        dist.all_gather_into_tensor(recv, send)                          # the single exchange
        e[2].record()
        hdr = recv.view(world, (cap + 1) * REC)[:, :4].contiguous().view(torch.int32).cpu()   # world ints: the counts
        counts = [int(x) for x in hdr.flatten()]
        ms_sum = 0.0
        for j in range(world):
            if j == rank:
                continue
            other = recv.data_ptr() + j * (cap + 1) * REC + REC
            ms = ctypes.c_double(0)
            r = L.cs_match(pts_ptr, n, other, counts[j], None, 0, ctypes.byref(ms))
            assert r == 0, L.cs_last_error()
            ms_sum += ms.value
        e[3].record()
        torch.cuda.synchronize()
        if rep > 0:
            t_ext.append(e[0].elapsed_time(e[1])); t_ag.append(e[1].elapsed_time(e[2])); t_match.append(ms_sum)
    med = [float(np.median(x)) for x in (t_ext, t_ag, t_match)]
    tot = reduce_max(dist, sum(med))
    ag = reduce_max(dist, med[1])
    ok = None
    if rank == 0:
        import oracle
        mine = np.frombuffer(send[REC:REC + n * REC].cpu().numpy().tobytes(), dtype=cs.SIFT_DTYPE)
        ok = True
        for j in range(1, min(world, 3)):
            off = j * (cap + 1) * REC + REC
            other = np.frombuffer(recv[off:off + counts[j] * REC].cpu().numpy().tobytes(), dtype=cs.SIFT_DTYPE)
            got, _ = cs.match_host(mine, other)
            want = oracle.match(mine, other, threads=8)
            ok = ok and bool(np.array_equal(want["match"], got["match"]) and np.array_equal(want["score"], got["score"]))
    return {"config": "all-pairs match, %d images 1920x1080, one per GPU (BASELINE config #5)" % world, "features": counts,
            "ms_extract": round(med[0], 4), "ms_allgather": round(ag, 4), "ms_match_%d_pairs_per_rank" % (world - 1): round(med[2], 4),
            "ms_total_max_over_ranks": round(tot, 4), "collectives": 1,
            "allgather_bytes_per_rank": (cap + 1) * REC, "capacity_records": cap, "check_vs_oracle": ok}


def cpu_baseline(imgs):
    """The oracle port (oracle/sift_oracle.c) on the host cores: one image per thread."""
    import oracle
    cores = os.cpu_count() or 1
    threads = min(cores, 32)
    per_thread = 8
    oracle.extract(imgs[0], OCTAVES, INIT_BLUR, THRESH)          # warm (loads the .so)

    def work(i):
        for j in range(per_thread):
            oracle.extract(imgs[(i + j) % len(imgs)], OCTAVES, INIT_BLUR, THRESH)
    t0 = time.perf_counter()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    [t.start() for t in ths]
    [t.join() for t in ths]
    dt = time.perf_counter() - t0
    n = threads * per_thread
    out = {"value": round(n / dt, 2), "unit": "images/s", "cores": threads, "kind": "port",
           "sample": "%d synthetic 1920x1080 images through oracle_extract (scalar C restatement), %d threads, %.1f s"
                     % (n, threads, dt)}
    out["opencv_sift"] = opencv_sift_baseline(imgs, cores)
    return out


def opencv_sift_baseline(imgs, cores, budget_s=6.0):
    """BASELINE.json's "scalar CPU OpenCV-SIFT baseline on the host cores, core count stated": a different
    algorithm variant (OpenCV's SIFT, 8-bit input), reported for orientation only; 1 thread, then all cores."""
    try:
        import cv2
    except Exception as e:                                    # not part of the contract: absent -> say so
        return {"unavailable": str(e)[:80]}
    im8 = [np.clip(np.rint(im), 0, 255).astype(np.uint8) for im in imgs[:4]]
    sift = cv2.SIFT_create(nOctaveLayers=5)
    res = {"host_cores": cores, "nOctaveLayers": 5}
    for name, nthreads in (("scalar", 1), ("all_cores", cores)):
        cv2.setNumThreads(nthreads)
        sift.detectAndCompute(im8[0], None)                   # warm
        t0, k, nk = time.perf_counter(), 0, 0
        while time.perf_counter() - t0 < budget_s / 2 and k < 64:
            kp, _ = sift.detectAndCompute(im8[k % len(im8)], None)
            nk += len(kp); k += 1
        dt = time.perf_counter() - t0
        res[name] = {"images_per_s": round(k / dt, 2), "threads": nthreads, "images": k, "features_per_image": round(nk / max(k, 1))}
    return res


# ------------------------------------------------------------------------------------------ reference arm
class RefSiftData(ctypes.Structure):
    _fields_ = [("numPts", ctypes.c_int), ("maxPts", ctypes.c_int), ("h_data", ctypes.c_void_p), ("d_data", ctypes.c_void_p)]


class RefCudaImage(ctypes.Structure):
    _fields_ = [("width", ctypes.c_int), ("height", ctypes.c_int), ("pitch", ctypes.c_int), ("h_data", ctypes.c_void_p),
                ("d_data", ctypes.c_void_p), ("t_data", ctypes.c_void_p), ("d_internalAlloc", ctypes.c_bool),
                ("h_internalAlloc", ctypes.c_bool)]


class quiet_stdout:
    """The reference printf()s on every call (quirk Q13): silence fd 1 meanwhile."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        self.null = os.open(os.devnull, os.O_WRONLY)
        os.dup2(self.null, 1)

    def __exit__(self, *a):
        try:
            ctypes.CDLL(None).fflush(None)
        except Exception:
            pass
        os.dup2(self.saved, 1)
        os.close(self.null)
        os.close(self.saved)


def load_cudart():
    for name in ("libcudart.so.12", "libcudart.so", "/usr/local/cuda/lib64/libcudart.so.12", "/usr/local/cuda/lib64/libcudart.so"):
        try:
            return ctypes.CDLL(name)
        except OSError:
            continue
    import glob
    for p in glob.glob(os.path.join(os.path.dirname(os.path.dirname(np.__file__)), "nvidia", "cuda_runtime", "lib", "libcudart.so*")):
        try:
            return ctypes.CDLL(p)
        except OSError:
            continue
    raise OSError("libcudart not found")


def run_reference(args):
    """The unmodified reference (oracle/_ref/libcudasift_ref.so, sm_100 build of Celebrandil/CudaSift) through its own
    C++ API.  This process never loads libcudasift_b200.so: the reference's own InitCuda / CudaImage::Download do the
    device work, libcudart (ctypes) only synchronises and uploads the match descriptors.  The reference has no CPU
    implementation of this path; if its library did not travel, the oracle port is timed on the host cores instead."""
    rank, world, local = dist_env()
    numa = bind_numa(local)
    imgs = make_images(rank, args.distinct, standalone=True)
    pitch = W if W % 128 == 0 else W - W % 128 + 128
    if not os.path.exists(REF_LIB):
        if rank == 0:
            cb = cpu_baseline(imgs)
            print(json.dumps({"impl": "reference", "metric": "1920x1080 images/sec ExtractSift", "value": cb["value"],
                              "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                              "higher_is_better": True, "scaling": "weak", "dtype": "f32", "data": "synthetic",
                              "config": workload_config(args.batch, len(imgs), pitch, 0, rounds_per_step(args)),
                              "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "images/s",
                                                          "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)
        return
    c = ctypes
    P = c.POINTER
    R = c.CDLL(REF_LIB, mode=c.RTLD_LOCAL)
    rt = load_cudart()
    rt.cudaMemcpy.argtypes = [c.c_void_p, c.c_void_p, c.c_size_t, c.c_int]
    init = R._Z8InitCudai; init.argtypes = [c.c_int]
    alloc = R._Z19AllocSiftTempMemoryiiib; alloc.restype, alloc.argtypes = c.c_void_p, [c.c_int, c.c_int, c.c_int, c.c_bool]
    extract = R._Z11ExtractSiftR8SiftDataR9CudaImageidffbPf
    extract.argtypes = [P(RefSiftData), P(RefCudaImage), c.c_int, c.c_double, c.c_float, c.c_float, c.c_bool, c.c_void_p]
    initdata = R._Z12InitSiftDataR8SiftDataibb; initdata.argtypes = [P(RefSiftData), c.c_int, c.c_bool, c.c_bool]
    freedata = R._Z12FreeSiftDataR8SiftData; freedata.argtypes = [P(RefSiftData)]
    match = R._Z13MatchSiftDataR8SiftDataS0_; match.restype, match.argtypes = c.c_double, [P(RefSiftData), P(RefSiftData)]
    imgalloc = R._ZN9CudaImage8AllocateEiiibPfS0_
    imgalloc.argtypes = [P(RefCudaImage), c.c_int, c.c_int, c.c_int, c.c_bool, c.c_void_p, c.c_void_p]
    imgdown = R._ZN9CudaImage8DownloadEv; imgdown.restype, imgdown.argtypes = c.c_double, [P(RefCudaImage)]
    with quiet_stdout():
        init(local)                      # one process per GPU: the reference keeps per-process state (quirk Q12)
    dist = init_dist(world, local)

    def sync_all():
        rt.cudaDeviceSynchronize()
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    B = args.batch
    images = []
    for i in range(B):
        im = RefCudaImage()
        arr = np.ascontiguousarray(imgs[i % len(imgs)], np.float32)
        imgalloc(c.byref(im), W, H, pitch, False, None, arr.ctypes.data_as(c.c_void_p))
        im._keep = arr
        imgdown(c.byref(im))
        images.append(im)
    sd = RefSiftData()
    initdata(c.byref(sd), MAX_PTS, True, True)
    tmp = alloc(W, H, OCTAVES, False)
    counts = [0] * B

    NR = rounds_per_step(args)      # passes per step (R is the reference library handle here)

    def step(download):
        for _ in range(NR):
            for i in range(B):
                if download:
                    imgdown(c.byref(images[i]))
                extract(c.byref(sd), c.byref(images[i]), OCTAVES, INIT_BLUR, THRESH, 0.0, False, tmp)
                counts[i] = sd.numPts
    sampler = ClockSampler(local)
    with quiet_stdout():
        for _ in range(max(1, args.warmup)):
            step(False)
        sync_all()
        sampler.start()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step(False)
        sync_all()
        dt = time.perf_counter() - t0
        clocks = sampler.stop()
        feats = float(np.mean(counts))
        t0 = time.perf_counter()
        esteps = max(1, args.steps // 2)
        for _ in range(esteps):
            step(True)
        sync_all()
        dte = time.perf_counter() - t0
    dt, dte = reduce_max(dist, dt), reduce_max(dist, dte)
    mres = None
    if rank == 0:
        synth_descriptors = synth_module(True).synth_descriptors
        mres = {}
        for n in (2000, 10000):
            s1, s2 = synth_descriptors(n, 1), synth_descriptors(n, 2)
            d1, d2 = RefSiftData(), RefSiftData()
            initdata(c.byref(d1), n + 64, True, True)      # +64: the reference writes past n1 (Q8)
            initdata(c.byref(d2), n + 64, False, True)
            d1.numPts = d2.numPts = n
            rt.cudaMemcpy(d1.d_data, s1.ctypes.data_as(c.c_void_p), s1.nbytes, 1)
            rt.cudaMemcpy(d2.d_data, s2.ctypes.data_as(c.c_void_p), s2.nbytes, 1)
            with quiet_stdout():
                ts = [match(c.byref(d1), c.byref(d2)) for _ in range(8)][2:]
            ms = float(np.median(ts))
            mres["n%d" % n] = {"ms": round(ms, 4), "gpair_per_s": round(n * n / (ms * 1e-3) / 1e9, 2)}
            freedata(c.byref(d1)); freedata(c.byref(d2))
        mres["how"] = "reference MatchSiftData (FindMaxCorr10), its own TimerGPU incl. the 5-field D2H copy"
    value = args.steps * B * NR * world / dt
    e2e = esteps * B * NR * world / dte
    if rank == 0:
        print(json.dumps({
            "impl": "reference", "metric": "1920x1080 images/sec ExtractSift", "value": round(value, 1),
            "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(dt / args.steps * 1e3, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(B, len(imgs), pitch, feats, NR),
            "api": "unmodified Celebrandil/CudaSift built for sm_100 (oracle/_ref), its own ExtractSift loop as in "
                   "mainSift.cpp:65-69, pre-allocated temp memory, one process per GPU; this process does not load libcudasift_b200.so",
            "clocks": clocks, "numa": numa,
            "cpu_baseline": {"value": round(value, 1), "unit": "images/s", "cores": 1, "kind": "reference",
                             "sample": "the reference is a CUDA library: timed on the GPU (1 host thread drives it), "
                                       "%d images" % (args.steps * B * NR)},
            "e2e": {"value": round(e2e, 1), "unit": "images/s", "h2d_bytes_per_step": B * NR * W * H * 4,
                    "d2h_bytes_per_step": int(B * NR * feats * REC),
                    "api": "CudaImage::Download + ExtractSift (host copy of the points included, cudaSiftH.cu:139-140)"},
            "match": mres,
        }), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="device-resident images per GPU (one pass over them = one round)")
    ap.add_argument("--rounds", type=int, default=0, help="passes over the images per step (0 = enough for a 0.3 s timed region)")
    ap.add_argument("--streams", type=int, default=2, help="batch extractors in flight (batch / streams images each)")
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic images per rank")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the keypoints of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the product computed; the reference arm has no dump")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_product(args)


if __name__ == "__main__":
    main()
