#!/usr/bin/env python
"""bench.py -- the BASELINE.json metric: PAF post-processing images/sec at 368x432.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the whole hot path (stages 1-5: bilinear x8 upsample materialising the
operator-surface tensors, Gaussian smoothing, 3x3 NMS peak extraction, PAF line-integral scoring,
greedy limb assignment + person assembly) over BATCHES_PER_STEP consecutive batches of 64 synthetic
368x432 images per GPU (BASELINE.json configs[1], batch 64; 32 batches make a step long enough --
about 12 ms -- for the clock and utilisation samplers to see the load).  Images shard across GPUs
with no data-path collective (weak scaling: every rank processes its own batches); the only exchange
is one final result gather.  One JSON line is printed by rank 0.

  value        images/s, whole job, inputs resident in HBM, timed with CUDA events (max over ranks)
  e2e          images/s through the host-buffer C-ABI entry (pinned host -> H2D -> kernels -> D2H of
               the result tables -> host arrays), copies inside the timed region; with the measured
               concurrent H2D ceiling of the box next to it
  roofline     the fused stage 1-3 kernel: algorithmic bytes (SURVEY.md 8d materialising contract)
               / its mean launch duration over the timed region
  configs      the other BASELINE.json configurations (656x368 x 256, crowded 1312x736 x 16, the
               non-materialising "lean" path, the reference's own front-end), each with stage times,
               a roofline and a check of sampled images against the oracle; configs[0] (CPU) and
               configs[4] (vgg2016 + this post-processing on the GPU) as context legs
  cpu_baseline the UNMODIFIED reference (its own Python byte-compiled into oracle/_ref/py + its C++
               compiled into oracle/_ref/libpaf_ref.so) on ONE host core on a bounded sample

--impl reference times that unmodified reference on all host cores (multiprocessing).
--dump-outputs DIR writes what the headline loop returned in its last step to DIR/<name>.npy (dump_outputs); the inputs
are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import importlib.util
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark only reads the tree it runs from (which may be read-only)

METRIC = "postprocess images/sec at 368x432"
UNIT = "images/s"
BATCH = 64              # images per batch (configs[1])
BATCHES_PER_STEP = int(os.environ.get("EKP_BENCH_BATCHES_PER_STEP", "32"))
H_LO, W_LO = 46, 54     # stride-8 map of a 368x432 image
PEOPLE = (1, 6)
INPUT_SETS = 4          # distinct input batches rotated between batches
N_CTX = int(os.environ.get("EKP_BENCH_CONTEXTS", "8"))   # contexts / CUDA streams the batches rotate over
N_CTX_CFG = int(os.environ.get("EKP_BENCH_CFG_CONTEXTS", "8"))   # ... in the configs[2] / configs[3] context legs


def algo_bytes(h, w, materialize=True):
    """SURVEY.md 8(d): materialising contract 4hw57 + 4HW57 per image; lean contract 4hw57."""
    return 4 * h * w * 57 + (4 * (8 * h) * (8 * w) * 57 if materialize else 0)


CONFIG = {
    "workload": "configs[1]: batch 64 synthetic heat(19ch)/PAF(38ch) at 46x54 stride-8 (368x432), "
                "dense front-end materialising heat_mat/paf_mat + PAF scoring + assembly",
    "batch": BATCH, "batches_per_step": BATCHES_PER_STEP, "images_per_step_per_gpu": BATCH * BATCHES_PER_STEP,
    "shape": "368x432", "people_per_image": "1-6", "frontend": "dense", "materialize": True,
    "pipelining": f"{N_CTX} contexts on {N_CTX} CUDA streams take the batches in turn (stages 4-5 of one batch overlap the "
                  "front-end kernel of the next); a repeated batch is one CUDA graph launch",
    "l2": "every batch writes 2.3 GB of operator-surface tensors (>> 126 MB L2); inputs rotate over "
          f"{INPUT_SETS} distinct batches",
}


def load_synthetic():
    """The synthetic generator WITHOUT importing the product package (which maps libekpose_b200.so): the reference
    arm must not have the product library in its process."""
    spec = importlib.util.spec_from_file_location("ekp_synthetic", os.path.join(ROOT, "torch_ekpose_b200", "synthetic.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def kernel_source_hash(name):
    with open(os.path.join(ROOT, "torch_ekpose_b200", "csrc", name), "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()[:16]


def ncu_constants():
    """Per-launch figures taken from the committed ncu captures (profiles/kernels.json): DRAM traffic of the roofline
    kernel, warp instructions of the latency / issue-bound ones.  Every entry carries the hash of the kernel source it
    was captured from; an entry whose source has changed since is REFUSED (reported as stale, value null)."""
    try:
        with open(os.path.join(ROOT, "profiles", "kernels.json")) as f:
            table = json.load(f)
    except Exception:
        return {}
    out = {}
    for key, ent in table.items():
        try:
            fresh = kernel_source_hash(ent["source"]) == ent["source_sha16"]
        except Exception:
            fresh = False
        out[key] = dict(ent, stale=not fresh)
    return out


# ---------------------------------------------------------------------------------------------
# clocks: NVML sampled in a thread DURING the timed regions (the same counters nvidia-smi prints)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._active = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            if self._active.is_set():
                try:
                    mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                    try:
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    self.samples.append(mhz)
                    for bit, name in self.REASONS.items():
                        if r & bit and name != "gpu_idle":
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def region(self, on: bool):
        (self._active.set if on else self._active.clear)()

    def stop(self):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=1)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------
# the reference's CPU path (checker code under oracle/, timed -- never shipped)
# ---------------------------------------------------------------------------------------------
_CPU = {}


def _cpu_setup():
    """Per process: the unmodified reference Python (oracle/_ref/py or /root/reference) over the compiled reference C++."""
    if "mod" not in _CPU:
        import oracle
        try:
            import cv2
            cv2.setNumThreads(1)   # one process = one core; the pool provides the parallelism
        except Exception:
            pass
        _CPU["oracle"] = oracle
        if oracle.have_ref() and (oracle.have_refpy() or os.path.isdir(oracle.REF_ROOT)):
            mod, cfg, impl = oracle.reference_python(use_ref=True)
            _CPU.update(mod=mod, cfg=cfg, impl=impl, kind="reference",
                        flavour="reference-python: UNMODIFIED lib/utils/paf_to_pose.py (paf_to_pose_cpp: NMS + cv2 nearest x8 of PAF and "
                                "heat + process_paf + getter loop) over the UNMODIFIED lib/pafprocess/pafprocess.cpp, both built "
                                "from /root/reference into oracle/_ref (bytecode / .so)")
        else:   # nothing of the reference could be built where this snapshot was made: the C restatements stand in
            _CPU.update(mod=None, cfg=None, impl=oracle.RefPaf() if oracle.have_ref() else oracle.PortPaf(), kind="port",
                        flavour="C restatements of NMS() and process_paf (oracle/frontend_oracle.c, oracle/paf_oracle.c)")
        _CPU["fe"] = oracle.Frontend()
    return _CPU


def cpu_reference_image(args):
    """paf_to_pose_cpp of the reference for one image (paf_to_pose.py:346-380)."""
    heat_hwc, paf_hwc = args
    c = _cpu_setup()
    if c["mod"] is not None:
        return len(c["mod"].paf_to_pose_cpp(heat_hwc, paf_hwc, c["cfg"]))
    return cpu_restatement_image(args)


def cpu_restatement_image(args):
    """The same path with the C restatement of NMS() in front of the compiled reference process_paf."""
    heat_hwc, paf_hwc = args
    c = _cpu_setup()
    fe, impl = c["fe"], c["impl"]
    peaks = fe.ref_nms(heat_hwc, np.float32(0.15))
    if len(peaks) == 0:
        return 0
    paf_up = fe.upsample_nearest(paf_hwc)
    heat_up = fe.upsample_nearest(heat_hwc)
    impl.process_paf(peaks[None], heat_up, paf_up)
    n = impl.get_num_humans()
    for hid in range(n):
        for part in range(18):
            cid = impl.get_part_cid(hid, part)
            if cid >= 0:
                impl.get_part_x(cid), impl.get_part_y(cid), impl.get_part_score(cid)
        impl.get_score(hid)
    return n


def cpu_dense_libs_image(args):
    """BASELINE.md section 4 "dense restatement": cv2.resize(INTER_LINEAR) + gaussian_filter + maximum_filter + reference
    process_paf -- the like-for-like CPU line of the dense GPU arm."""
    c = _cpu_setup()
    return c["oracle"].dense_restatement_libs(args[0], args[1], c["impl"])[1]


def timed_loop(fn, images, budget_s):
    """One core, bounded: loops over the sample images until ~budget_s of CPU work is done."""
    t0 = time.perf_counter()
    done = 0
    while True:
        for hw in images:
            fn(hw)
            done += 1
            if time.perf_counter() - t0 > budget_s:
                break
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return done / dt, done, dt


def hwc_images(heat_nchw, paf_nchw, count):
    return [(np.ascontiguousarray(heat_nchw[i].transpose(1, 2, 0)), np.ascontiguousarray(paf_nchw[i].transpose(1, 2, 0)))
            for i in range(min(count, len(heat_nchw)))]


def host_cores():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_baseline_block(sample_imgs, budget_s):
    """cpu_baseline of the product arm: ONE core; the reference itself plus two labelled context numbers."""
    c = _cpu_setup()
    v, done, dt = timed_loop(cpu_reference_image, sample_imgs, budget_s)
    v2, d2, t2 = timed_loop(cpu_restatement_image, sample_imgs, min(3.0, budget_s / 3))
    v3, d3, t3 = timed_loop(cpu_dense_libs_image, sample_imgs[:4], min(4.0, budget_s / 2))
    return {"value": v, "unit": UNIT, "cores": 1, "kind": c["kind"], "flavour": c["flavour"],
            "sample": f"{done} images ({dt:.1f} s) of the same synthetic 368x432 workload (configs[1] scenes, 1-6 people) on 1 core",
            "other": {
                "c_restatement_of_reference_frontend_images_per_s": {
                    "value": v2, "cores": 1, "sample": f"{d2} images ({t2:.1f} s): oracle/frontend_oracle.c NMS + nearest x8 + reference process_paf"},
                "dense_restatement_library_primitives_images_per_s": {
                    "value": v3, "cores": 1,
                    "sample": f"{d3} images ({t3:.1f} s): cv2.resize(INTER_LINEAR) x8 + scipy gaussian_filter(sigma 3) + maximum_filter(3) + "
                              "reference process_paf (BASELINE.md section 4; the CPU form of what the dense GPU arm computes)"}}}


def c1_cpu_leg():
    """configs[0]: the reference's vgg2016 (random init, torch.manual_seed(0)) CPU forward on one 368x432 input + the
    reference's paf_to_pose_cpp on one synthetic 46x54 scene (the random-init network's heat maps stay below the
    0.15 threshold, SURVEY.md 8d, so the post-processing is timed on the synthetic maps of the same shape)."""
    import torch
    c = _cpu_setup()
    if c["mod"] is None:
        return {"unavailable": "oracle/_ref/py absent"}
    syn = load_synthetic()
    vgg = c["oracle"].reference_module("lib.network.vgg2016")
    torch.manual_seed(0)
    devnull = open(os.devnull, "w")
    old = sys.stdout
    sys.stdout = devnull          # the reference prints while it builds the network
    try:
        net = vgg.OpenPose().eval()
    finally:
        sys.stdout = old
        devnull.close()
    x = torch.randn(1, 3, 368, 432)
    with torch.no_grad():
        net(x)
        t0 = time.perf_counter()
        (paf, heat), _ = net(x)
        fwd = time.perf_counter() - t0
    hw, pw = syn.make_scene(H_LO, W_LO, 3, 1)
    c["mod"].paf_to_pose_cpp(hw, pw, c["cfg"])
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        humans = c["mod"].paf_to_pose_cpp(hw, pw, c["cfg"])
    post = (time.perf_counter() - t0) / reps
    return {"workload": "configs[0]: vgg2016 random-init forward + reference paf_to_pose_cpp, one 368x432 image, CPU",
            "forward_ms": 1000 * fwd, "forward_threads": torch.get_num_threads(), "output_shapes": [list(paf.shape), list(heat.shape)],
            "random_init_heat_max": float(heat.max()), "postprocess_ms": 1000 * post, "humans": len(humans),
            "frames_per_s": 1.0 / (fwd + post)}


def run_reference_arm(args, rank, world):
    """The UNMODIFIED reference on all host cores (rank 0 only; the other ranks exit without work)."""
    if rank != 0:
        return
    import multiprocessing as mp

    import oracle
    oracle.build()
    syn = load_synthetic()
    heat, paf = syn.make_batch(BATCH, H_LO, W_LO, PEOPLE, seed=100)
    imgs = hwc_images(heat, paf, BATCH)
    cores = host_cores()
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        # calibrate, then bound the per-step sample so that warmup + steps end within ~2 minutes
        pool.map(cpu_reference_image, imgs[:cores], chunksize=1)
        t0 = time.perf_counter()
        pool.map(cpu_reference_image, imgs, chunksize=max(1, BATCH // (cores * 2)))
        rate = BATCH / (time.perf_counter() - t0)
        per_step = int(max(cores, min(BATCH * BATCHES_PER_STEP, 90.0 * rate / max(args.steps + args.warmup, 1))))
        sample = [imgs[i % BATCH] for i in range(per_step)]
        chunk = max(1, per_step // (cores * 4))
        for _ in range(args.warmup):
            pool.map(cpu_reference_image, sample, chunksize=chunk)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            pool.map(cpu_reference_image, sample, chunksize=chunk)
        dt = time.perf_counter() - t0
        value = per_step * args.steps / dt
        # context numbers on the same pool: the C restatement of the reference front-end, and the dense restatement
        t0 = time.perf_counter()
        pool.map(cpu_restatement_image, imgs, chunksize=max(1, BATCH // (cores * 2)))
        v_c = BATCH / (time.perf_counter() - t0)
        nd = max(cores, 16)
        t0 = time.perf_counter()
        pool.map(cpu_dense_libs_image, [imgs[i % BATCH] for i in range(nd)], chunksize=1)
        v_d = nd / (time.perf_counter() - t0)
    c = _cpu_setup()
    sample_txt = (f"{args.steps} steps x {per_step} images of configs[1] (the 64 synthetic scenes of the product arm's first input set, "
                  f"cycled) on {cores} processes, one per host core in this process's affinity mask")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": CONFIG,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": c["kind"], "flavour": c["flavour"], "sample": sample_txt,
                             "value_per_core": value / cores,
                             "other": {"c_restatement_of_reference_frontend_images_per_s": {"value": v_c, "cores": cores},
                                       "dense_restatement_library_primitives_images_per_s": {"value": v_d, "cores": cores}}},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# the product arm
# ---------------------------------------------------------------------------------------------
def pin_rank(local_rank, local_world):
    """A disjoint slice of the host cores per rank (before any pinned allocation): the ranks' submission threads and
    their pinned buffers do not migrate over each other."""
    if not hasattr(os, "sched_setaffinity") or local_world <= 1:
        return sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else []
    cores = sorted(os.sched_getaffinity(0))
    per = max(1, len(cores) // local_world)
    mine = cores[local_rank * per:(local_rank + 1) * per] or cores
    try:
        os.sched_setaffinity(0, mine)
    except OSError:
        return cores
    return mine


class Runner:
    """N_CTX contexts on N_CTX streams taking batches of one configuration in turn."""

    def __init__(self, ek, torch, dev, local_rank, n, h, w, people, seed, max_peaks, max_humans, max_part, max_cand, nctx=N_CTX, nsets=INPUT_SETS,
                 mat_nctx=None):
        self.ek, self.torch, self.dev = ek, torch, dev
        self.mat_nctx = min(nctx, mat_nctx or nctx)   # contexts the MATERIALISING batches rotate over (each holds n x 65 x the input bytes)
        self.n, self.h, self.w = n, h, w
        self.syn = load_synthetic()
        self.host, self.devs = [], []
        for s in range(nsets):
            heat, paf = self.syn.make_batch(n, h, w, people, seed=seed + s)
            self.host.append((heat, paf))
            self.devs.append((torch.from_numpy(heat).to(dev), torch.from_numpy(paf).to(dev)))
        self.pps = [ek.PostProcessor(device=local_rank, max_batch=n, max_h=h, max_w=w, max_peaks=max_peaks, max_humans=max_humans,
                                     max_part=max_part, max_cand=max_cand) for _ in range(nctx)]
        self.streams = [torch.cuda.Stream(dev) for _ in range(nctx)]
        self.main = torch.cuda.current_stream(dev)

    def submit(self, i, frontend, materialize, inputs=None):
        k = i % (self.mat_nctx if materialize else len(self.pps))
        hd, pd = (inputs or self.devs)[i % len(self.devs)]
        self.pps[k].run(hd, pd, layout="nchw", frontend=frontend, materialize=materialize, stream=self.streams[k])

    def fork(self):
        for s_ in self.streams:
            s_.wait_stream(self.main)

    def join(self):
        for s_ in self.streams:
            self.main.wait_stream(s_)

    def throughput(self, frontend, materialize, batches, warm=None):
        torch = self.torch
        for i in range(warm if warm is not None else 2 * len(self.pps)):
            self.submit(i, frontend, materialize)
        torch.cuda.synchronize(self.dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(self.main)
        self.fork()
        for i in range(batches):
            self.submit(i, frontend, materialize)
        self.join()
        b.record(self.main)
        torch.cuda.synchronize(self.dev)
        ms = a.elapsed_time(b)
        return self.n * batches / (ms / 1000.0), ms / batches

    def isolated_stage_ms(self, frontend, materialize, runs=24):
        """One context, one stream, nothing overlapping: device time per stage (events recorded by the library)."""
        pp = self.pps[0]
        self.torch.cuda.synchronize(self.dev)
        pp.set_timing(True)
        for i in range(runs):
            hd, pd = self.devs[i % len(self.devs)]
            pp.run(hd, pd, layout="nchw", frontend=frontend, materialize=materialize, stream=self.streams[0])
        pp.results()
        ms, _ = pp.stage_times()
        pp.set_timing(False)
        return ms

    def oracle_check(self, frontend, materialize, samples=2):
        """Sampled images of input set 0 through the product path and through the oracle (the CHECKER): subset rows must
        agree bit for bit (front-end restatement of oracle/frontend_oracle.c + the compiled reference process_paf)."""
        import oracle
        fe = oracle.Frontend()
        impl = oracle.RefPaf() if oracle.have_ref() else oracle.PortPaf()
        pp = self.pps[0]
        hd, pd = self.devs[0]
        pp.run(hd, pd, layout="nchw", frontend=frontend, materialize=materialize, stream=self.streams[0])
        res = pp.results()
        heat, paf = self.host[0]
        idx = sorted({0, self.n // 2, self.n - 1})[:samples] if samples < 3 else sorted({0, self.n // 3, self.n // 2, self.n - 1})[:samples]
        ok, humans = True, 0
        for i in idx:
            hw = np.ascontiguousarray(heat[i].transpose(1, 2, 0))
            pw = np.ascontiguousarray(paf[i].transpose(1, 2, 0))
            if frontend == "dense":
                peaks, paf_mat = fe.dense_peaks(hw), fe.upsample_bilinear(pw)
            else:
                peaks, paf_mat = fe.ref_nms(hw), fe.upsample_nearest(pw)
            sub, _ = oracle.subset_of(impl, peaks, 8 * self.h, 8 * self.w, paf_mat)
            n = int(res["num_humans"][i])
            same = n == len(sub) and np.array_equal(res["subset"][i, :n].view(np.uint32), sub.view(np.uint32)) and \
                int(res["n_peaks"][i]) == len(peaks)
            ok = ok and bool(same)
            humans += n
        return {"images_checked": [int(i) for i in idx], "humans": humans, "bit_exact_vs_oracle": ok,
                "oracle": "oracle/frontend_oracle.c front-end + " + ("oracle/_ref/libpaf_ref.so (compiled reference)" if oracle.have_ref() else "oracle/paf_oracle.c")}

    def launches(self):
        return sum(p.kernel_launches() for p in self.pps), sum(p.graph_launches() for p in self.pps)

    def close(self):
        for p in self.pps:
            p.close()
        self.pps, self.devs = [], []
        self.torch.cuda.empty_cache()


DUMP_MAT_POSITIONS = 256   # (y, x) positions per image sampled from heat_mat / paf_mat (2.3 GB per batch in full)
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, R, nb):
    """What the timed headline loop handed its caller in its last step, as DIR/<name>.npy (float32 / float64), so that two
    builds can be compared output for output.  Every context still holds the batch it ran last, so the last
    min(contexts, batches per step) batches of the step are read back, as many of them as fit DUMP_LIMIT_BYTES: their
    result tables (rows past num_humans / n_peaks zeroed) and the operator-surface tensors at a fixed, seeded sample of
    positions.  Dumped batches are stacked along a leading axis, the oldest first."""
    torch = R.torch
    pp0 = R.pps[0]
    per_batch = R.n * (8 * (3 + 19) + 4 * (20 * pp0.max_humans + 4 * pp0.max_peaks + 57 * DUMP_MAT_POSITIONS))
    fit = (DUMP_LIMIT_BYTES - 16 * DUMP_MAT_POSITIONS) // per_batch
    batches = range(nb - max(1, min(BATCHES_PER_STEP, R.mat_nctx, nb, fit)), nb)
    rng = np.random.default_rng(0)
    ys = torch.from_numpy(rng.integers(0, 8 * R.h, DUMP_MAT_POSITIONS)).to(R.dev)
    xs = torch.from_numpy(rng.integers(0, 8 * R.w, DUMP_MAT_POSITIONS)).to(R.dev)
    cols = {k: [] for k in ("num_humans", "n_peaks", "overflow", "subset", "peaks", "part_off", "heat_mat_sample", "paf_mat_sample")}
    for i in batches:
        pp = R.pps[i % R.mat_nctx]
        res = pp.results(with_peaks=True, raise_on_overflow=False)
        subset = res["subset"].copy()
        peaks = np.stack([res["peaks"][f].astype(np.float32) for f in ("x", "y", "score", "id")], axis=-1)
        for j in range(len(subset)):
            subset[j, int(res["num_humans"][j]):] = 0
            peaks[j, int(res["n_peaks"][j]):] = 0
        for k in ("num_humans", "n_peaks", "overflow", "part_off"):
            cols[k].append(res[k].astype(np.float64))
        cols["subset"].append(subset)
        cols["peaks"].append(peaks)
        cols["heat_mat_sample"].append(pp.heat_mat[:, ys, xs, :].cpu().numpy())
        cols["paf_mat_sample"].append(pp.paf_mat[:, ys, xs, :].cpu().numpy())
    arrays = {k: np.stack(v) for k, v in cols.items()}
    arrays["mat_sample_yx"] = np.stack([ys.cpu().numpy(), xs.cpu().numpy()], axis=1).astype(np.float64)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, f"dump of {total} bytes exceeds {DUMP_LIMIT_BYTES}"
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


FRONTEND_KERNELS = {("dense", True): ["dense_frontend_kernel<mat>"], ("dense", False): ["dense_plane_kernel"],
                    ("reference", False): ["ref_scan_kernel", "ref_refine_kernel"]}
STAGE_BOUNDS = {
    "peak_sort": ("peaks_sort_kernel", "latency: one short block per 256 peaks (histogram, scatter, rank within the part's bucket)"),
    "connect": ("paf_connect_kernel", "latency / occupancy: one block per (limb, image) walks stage, score, compact, sort, assign; "
                                      "gathers from L2: ten lanes per pair (ordinary scenes) or one thread per pair in two exact passes (crowds)"),
    "assemble": ("assemble_kernel", "latency: the 19 limbs of an image are a serial chain (one warp per image; float sums in limb order)"),
}


def issue_model(ents, kernel_ms, sm_mhz):
    """achieved warp instructions / s against 148 SMs x 4 issue slots x the SM clock (instruction counts from the committed
    ncu capture; refused when the kernel source changed since)."""
    missing = sum(e is None for e in ents)
    ents = [e for e in ents if e is not None]
    if not ents:
        return {"unavailable": "no ncu capture of this kernel / configuration in profiles/kernels.json"}
    if any(e["stale"] for e in ents):
        return {"stale": True, "reason": f"{ents[0]['source']} changed since {ents[0].get('capture')} was captured"}
    inst = sum(e["warp_instructions_per_launch"] for e in ents)
    out = {"warp_instructions_per_launch": inst, "issue_active_pct_under_ncu": [e["issue_active_pct"] for e in ents],
           "source": ents[0].get("capture")}
    if missing:
        out["note"] = f"{missing} of the stage's kernels has no capture: a lower bound"
    if sm_mhz and kernel_ms > 0:
        ipeak = 148 * 4 * sm_mhz * 1e6
        out.update(achieved_ginst_s=inst / (kernel_ms / 1e3) / 1e9, peak_ginst_s=ipeak / 1e9, frac=inst / (kernel_ms / 1e3) / ipeak)
    return out


def roofline_entry(frontend, n, h, w, materialize, stage_ms, peak, peak_src, consts, sm_mhz=None):
    """Rooflines of one configuration.  The front-end kernel is HBM-bound when it materialises the operator-surface
    tensors; without them it moves 65x fewer bytes and is bound by instruction issue.  Stages 4-5 are short latency-bound
    kernels: their issue fraction says how far from ANY throughput bound they run."""
    shape = f"{8 * h}x{8 * w}x{n}"
    mode = f"{frontend}_{'mat' if materialize else 'lean'}"
    kernels = FRONTEND_KERNELS.get((frontend, materialize)) or FRONTEND_KERNELS[(frontend, False)]
    kernel_ms = stage_ms["frontend"]
    ab = algo_bytes(h, w, materialize) * n
    achieved = ab / (kernel_ms / 1000.0) / 1e9 if kernel_ms > 0 else None
    ents = [consts.get(f"{k}|{shape}|{mode}") for k in kernels]
    out = {"kernel": " + ".join(kernels), "bound": "hbm" if materialize and frontend == "dense" else "issue",
           "algorithmic_bytes_per_launch": ab, "kernel_ms": kernel_ms, "achieved": achieved, "peak": peak, "unit": "GB/s",
           "frac": achieved / peak if achieved else None, "peak_source": peak_src}
    if out["bound"] == "hbm":
        e = ents[0]
        out["traffic"] = e["dram_bytes_per_launch"] if e and not e["stale"] else None
    else:
        out["note"] = "HBM fraction is small by construction (nothing full-resolution is written); the bound is instruction issue: see `issue`"
        out["issue"] = issue_model(ents, kernel_ms, sm_mhz)
    stages = {}
    for st, (kname, why) in STAGE_BOUNDS.items():
        stages[st] = {"kernel": kname, "ms": stage_ms[st], "bound": why, "issue": issue_model([consts.get(f"{kname}|{shape}|{mode}")], stage_ms[st], sm_mhz)}
    out["stages_4_5"] = stages
    return out


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", world))
    my_cores = pin_rank(local_rank, local_world)

    import torch_ekpose_b200 as ek

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL may print its version banner on stdout when the communicator is created; stdout must
        # carry exactly one JSON line, so fd 1 points at stderr while the communicator comes up.
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

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    steps, warmup = args.steps, max(args.warmup, 3)
    consts = ncu_constants()
    peak, peak_src = measured_peak()
    clocks = ClockSampler(local_rank)
    clocks.start()

    # ---- headline: configs[1], dense front-end, materialising ---------------------------------------------------
    R = Runner(ek, torch, dev, local_rank, BATCH, H_LO, W_LO, PEOPLE, seed=100 + 17 * rank, max_peaks=1024, max_humans=32,
               max_part=64, max_cand=512)
    stream = R.main
    nb = steps * BATCHES_PER_STEP
    for i in range(warmup * BATCHES_PER_STEP):
        R.submit(i, "dense", True)
    for p_ in R.pps:
        p_.results()
    l0, g0 = R.launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    clocks.region(True)
    ev0.record(stream)
    R.fork()
    for i in range(nb):
        R.submit(i, "dense", True)
    R.join()
    ev1.record(stream)
    barrier()
    clocks.region(False)
    ms = ev0.elapsed_time(ev1)
    l1, g1 = R.launches()
    launches, graph_batches = l1 - l0, g1 - g0
    res = R.pps[(nb - 1) % N_CTX].results()
    total_humans = int(res["num_humans"].sum())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, R, nb)
    iso_ms = R.isolated_stage_ms("dense", True)
    c2_check = R.oracle_check("dense", True) if rank == 0 else None

    # ---- e2e: host buffers through the C ABI, copies in the timed region ---------------------------------------
    # A stream of batches the way a caller would drive it: every batch's inputs come from pinned host memory (one block
    # per batch: heat directly followed by PAF, so the library moves it with ONE copy) and every batch's result tables are
    # read back on the host inside the timed region; N_CTX contexts keep the H2D of batch i+1 under the kernels of batch i.
    pinned = []
    for s in range(INPUT_SETS):
        pb = ek.PinnedBatch(BATCH, H_LO, W_LO, "nchw", write_combined=bool(int(os.environ.get("EKP_BENCH_WC", "0"))))
        np.copyto(pb.heat, R.host[s][0])
        np.copyto(pb.paf, R.host[s][1])
        pinned.append(pb)
    pin_inputs = [(pb.heat, pb.paf) for pb in pinned]

    def e2e_loop(batches):
        got = None
        for i in range(batches):
            if i >= N_CTX:
                got = R.pps[i % N_CTX].human_tables()      # results of batch i-N_CTX (waits for it)
            R.submit(i, "dense", True, inputs=pin_inputs)
        for i in range(max(batches - N_CTX, 0), batches):
            got = R.pps[i % N_CTX].human_tables()
        return got

    e2e_loop(2 * N_CTX)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    clocks.region(True)
    t_wall = time.perf_counter()
    e0.record(stream)
    R.fork()
    e2e_loop(nb)
    R.join()
    e1.record(stream)
    barrier()
    clocks.region(False)
    e2e_wall_ms = 1000.0 * (time.perf_counter() - t_wall)
    e2e_ms = max(e0.elapsed_time(e1), 0.0)
    h2d = BATCH * H_LO * W_LO * 57 * 4
    pp0 = R.pps[0]
    d2h = int(BATCH * (((16 + (80 + 16 * 18 + 4) * pp0.max_humans) + 15) // 16) * 16)   # one packed record per image

    # ---- the box's concurrent H2D ceiling: every rank copies the same 36 MB blocks at the same time --------------
    hd_dst = [torch.empty(pinned[0].nbytes, dtype=torch.uint8, device=dev) for _ in range(N_CTX)]
    pin_t = [torch.empty(pinned[0].nbytes, dtype=torch.uint8).pin_memory() for _ in range(N_CTX)]

    def h2d_round(reps):
        for r_ in range(reps):
            for k in range(N_CTX):
                with torch.cuda.stream(R.streams[k]):
                    hd_dst[k].copy_(pin_t[k], non_blocking=True)
    h2d_round(4)
    reps = 8
    h2d_ceiling = 0.0
    for _ in range(3):   # best of three rounds: a ceiling
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream)
        R.fork()
        h2d_round(reps)
        R.join()
        c1.record(stream)
        barrier()
        h2d_ceiling = max(h2d_ceiling, pinned[0].nbytes * reps * N_CTX / (c0.elapsed_time(c1) / 1e3) / 1e9)
    del hd_dst, pin_t

    clk = clocks.stop()

    # ---- context: the same batch on the non-materialising path, both front-ends -----------------------------------
    configs = {}

    def measure(run, name, workload, frontend, materialize, batches, check):
        barrier()   # every rank measures the same leg at the same time (a rank still in its previous phase disturbs the host side of the others)
        ips, ms_b = run.throughput(frontend, materialize, batches)
        st = run.isolated_stage_ms(frontend, materialize)
        ent = {"workload": workload, "contexts": run.mat_nctx if materialize else len(run.pps), "images_per_s_per_gpu": ips, "ms_per_batch_pipelined": ms_b, "stage_ms_isolated": st,
               "stages_4_5_ms_isolated": st["peak_sort"] + st["connect"] + st["assemble"],
               "roofline": roofline_entry(frontend, run.n, run.h, run.w, materialize, st, peak, peak_src, consts, clk.get("sm_mhz"))}
        if check and rank == 0:
            ent["oracle_check"] = run.oracle_check(frontend, materialize)
        configs[name] = ent

    measure(R, "c2_368x432_x64_dense_lean", "configs[1] shapes, dense front-end, nothing full-resolution written (the deployment path)", "dense", False, 200, True)
    measure(R, "c2_368x432_x64_reference_lean", "configs[1] shapes, the reference's own front-end (stride-8 NMS + bicubic refinement)", "reference", False, 200, True)
    for pb in pinned:
        pb.close()
    R.close()

    if not args.headline_only:
        # configs[2]: 656x368 frames, batch 256
        R3 = Runner(ek, torch, dev, local_rank, 256, 46, 82, (2, 8), seed=300 + 7 * rank, max_peaks=1024, max_humans=32, max_part=64,
                    max_cand=512, nctx=N_CTX_CFG, nsets=2, mat_nctx=4)
        measure(R3, "c3_656x368_x256_dense_materialised", "configs[2]: 656x368, batch 256, dense front-end + operator-surface tensors", "dense", True, 12, True)
        measure(R3, "c3_656x368_x256_dense_lean", "configs[2] without materialisation", "dense", False, 40, False)
        measure(R3, "c3_656x368_x256_reference_lean", "configs[2], reference front-end", "reference", False, 40, True)
        c3_host = R3.host[0]
        R3.close()
        # configs[3]: crowded 1312x736, 30-40 people, batch 16
        R4 = Runner(ek, torch, dev, local_rank, 16, 92, 164, (30, 40), seed=400 + 7 * rank, max_peaks=2048, max_humans=128, max_part=128,
                    max_cand=1024, nctx=N_CTX_CFG, nsets=2, mat_nctx=4)
        measure(R4, "c4_1312x736_x16_crowded_dense_materialised", "configs[3]: 1312x736, 30-40 people, batch 16, dense front-end + operator-surface tensors", "dense", True, 30, True)
        measure(R4, "c4_1312x736_x16_crowded_dense_lean", "configs[3] without materialisation", "dense", False, 60, True)
        measure(R4, "c4_1312x736_x16_crowded_reference_lean", "configs[3], reference front-end", "reference", False, 60, True)
        R4.close()

        # configs[2] as named: the 256-frame batch SHARDED over the ranks (strong scaling), results gathered with NCCL
        from torch_ekpose_b200 import sharding
        syn = load_synthetic()
        gheat, gpaf = syn.make_batch(256, 46, 82, (2, 8), seed=300)   # the same global batch on every rank
        lo, hi = sharding.shard_bounds(256, world, rank)
        spp = ek.PostProcessor(device=local_rank, max_batch=hi - lo, max_h=46, max_w=82, max_peaks=1024, max_humans=32, max_part=64, max_cand=512)
        sh, sp = torch.from_numpy(gheat[lo:hi]).to(dev), torch.from_numpy(gpaf[lo:hi]).to(dev)
        for _ in range(3):
            spp.run(sh, sp, frontend="dense", materialize=True)
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        reps3 = 10
        for _ in range(reps3):
            spp.run(sh, sp, frontend="dense", materialize=True)
        s1.record(stream)
        barrier()
        shard_ms = s0.elapsed_time(s1) / reps3
        spp.close()
        del sh, sp
        torch.cuda.empty_cache()
        # the library's own sharded entry (host arrays in, gathered tables out on every rank)
        t0 = time.perf_counter()
        gnum, gsub = sharding.postprocess_sharded(gheat, gpaf, frontend="dense", materialize=False, max_humans=32, max_peaks=1024)
        gather_s = time.perf_counter() - t0
        tt = torch.tensor([shard_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        shard_ms = float(tt[0])
        ent = {"workload": f"configs[2]: ONE 656x368 batch of 256 frames sharded over {world} GPU(s) ({hi - lo} frames on rank 0), dense front-end + "
                           "operator-surface tensors, max over ranks",
               "ms_per_global_batch": shard_ms, "images_per_s_whole_job": 256 / (shard_ms / 1e3), "scaling": "strong",
               "postprocess_sharded": {"humans_total": int(gnum.sum()), "gathered_rows": int(len(gnum)), "wall_s_incl_context_setup": gather_s}}
        if rank == 0:
            import oracle
            fe, impl = oracle.Frontend(), (oracle.RefPaf() if oracle.have_ref() else oracle.PortPaf())
            okc = True
            for i in (0, 255):   # first image of the first shard, last image of the last shard
                hw = np.ascontiguousarray(gheat[i].transpose(1, 2, 0)); pw = np.ascontiguousarray(gpaf[i].transpose(1, 2, 0))
                sub, _ = oracle.subset_of(impl, fe.dense_peaks(hw), 368, 656, fe.upsample_bilinear(pw))
                okc = okc and int(gnum[i]) == len(sub) and np.array_equal(gsub[i, :len(sub)].view(np.uint32), sub.view(np.uint32))
            ent["postprocess_sharded"]["bit_exact_vs_oracle_images_0_255"] = bool(okc)
        configs["c3_656x368_x256_sharded"] = ent

        # configs[4]: the reference's vgg2016 (unmodified, random init) on cuDNN feeding the post-processing on the same GPU
        try:
            configs["c5_vgg2016_plus_postprocess"] = c5_leg(ek, torch, dist, dev, local_rank, rank, world, barrier)
        except Exception as e:   # never lose the headline to a context leg
            configs["c5_vgg2016_plus_postprocess"] = {"unavailable": f"{type(e).__name__}: {e}"}

    # ---- max over ranks, final result gather -------------------------------------------------------
    t = torch.tensor([ms, e2e_ms, e2e_wall_ms, float(total_humans), h2d_ceiling], dtype=torch.float64, device=dev)
    h2d_all = [h2d_ceiling]
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        gathered = [torch.zeros(BATCH, dtype=torch.int32, device=dev) for _ in range(world)]
        dist.all_gather(gathered, torch.from_numpy(res["num_humans"]).to(dev))   # the final result gather
        total_humans = int(sum(int(g.sum()) for g in gathered))
        ms, e2e_ms, e2e_wall_ms = float(tmax[0]), float(tmax[1]), float(tmax[2])
        hl = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(hl, t[4:5].contiguous())
        h2d_all = [float(x[0]) for x in hl]

    if rank == 0:
        images = BATCH * nb * world
        value = images / (ms / 1000.0)
        # Roofline of the dominant kernel (fused stages 1-3).  The batches are pipelined over N_CTX streams, so per-kernel
        # event intervals overlap each other; the honest per-launch duration over the timed region is
        # (timed region) / (launches of that kernel), which also charges the kernel for everything else in the step (a lower
        # bound on its bandwidth).  kernel_ms_isolated is the same kernel timed alone (library events, one stream).
        per_launch_ms = ms / nb
        ab = algo_bytes(H_LO, W_LO) * BATCH
        achieved = ab / (per_launch_ms / 1000.0) / 1e9
        traffic_ent = consts.get("dense_frontend_kernel<mat>|368x432x64|dense_mat")
        traffic = traffic_ent["dram_bytes_per_launch"] if traffic_ent and not traffic_ent["stale"] else None
        e2e_val = images / (max(e2e_ms, e2e_wall_ms) / 1000.0)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": CONFIG,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic,
                         "traffic_note": None if traffic else ("profiles/kernels.json entry is stale: dense_frontend.cu changed since the capture" if traffic_ent else "no capture"),
                         "kernel": "dense_frontend_kernel (stages 1-3 fused, materialising)",
                         "kernel_ms": per_launch_ms, "kernel_ms_isolated": iso_ms["frontend"],
                         "frac_isolated": ab / (iso_ms["frontend"] / 1000.0) / 1e9 / peak if iso_ms["frontend"] > 0 else None,
                         "algorithmic_bytes_per_launch": ab, "peak_source": peak_src, "launches_averaged": nb},
            "stage_ms_isolated": iso_ms, "oracle_check": c2_check,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d * BATCHES_PER_STEP, "d2h_bytes_per_step": d2h * BATCHES_PER_STEP,
                    "device_ms_per_step": e2e_ms / steps, "wall_ms_per_step": e2e_wall_ms / steps,
                    "h2d_gbs_achieved_whole_job": e2e_val * (h2d / BATCH) / 1e9,
                    "h2d_ceiling_gbs_sum_of_gpus": sum(h2d_all), "h2d_ceiling_gbs_per_gpu": h2d_all,
                    # every rank moves the same bytes per step and the step ends with the slowest rank (max over ranks), so the
                    # ceiling of THIS metric is N x the slowest GPU's concurrent H2D rate, not the sum
                    "h2d_ceiling_gbs_equal_work": min(h2d_all) * world,
                    "frac_of_h2d_ceiling": e2e_val * (h2d / BATCH) / 1e9 / (min(h2d_all) * world) if min(h2d_all) > 0 else None,
                    "h2d_ceiling_how": f"all ranks at once: {N_CTX} streams x 8 copies of one {h2d} B pinned block each (the same copy the e2e path issues per batch), best of 3 rounds",
                    "api": f"ekp_postprocess_host + ekp_results_humans; one pinned block per batch (heat|paf, ONE H2D copy); {N_CTX} contexts / "
                           f"{N_CTX} streams so the H2D of one batch overlaps the kernels of the previous one; rank pinned to cores {my_cores[:1]}..{my_cores[-1:]}"},
            "gpu_launches": int(launches), "cuda_graph_batches": int(graph_batches), "clocks": clk,
            "humans_found_last_batch": total_humans, "configs": configs,
        }
        if world == 1 and not args.no_cpu_baseline:
            import oracle
            oracle.build()
            syn = load_synthetic()
            heat, paf = syn.make_batch(16, H_LO, W_LO, PEOPLE, seed=100)
            line["cpu_baseline"] = cpu_baseline_block(hwc_images(heat, paf, 16), args.cpu_seconds)
            try:
                configs["c1_cpu_vgg2016_plus_reference_postprocess"] = c1_cpu_leg()
            except Exception as e:
                configs["c1_cpu_vgg2016_plus_reference_postprocess"] = {"unavailable": f"{type(e).__name__}: {e}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def c5_leg(ek, torch, dist, dev, local_rank, rank, world, barrier):
    """configs[4]: end-to-end vgg2016 inference.  The reference's OWN network (lib/network/vgg2016.py, unmodified bytecode
    from oracle/_ref/py, random init with torch.manual_seed(0)) runs on cuDNN through PyTorch; frames are uploaded as
    uint8, padded + normalised by the input-side kernel (estimator.py:52-68 geometry), and the network's outputs go to the
    CUDA post-processing without leaving the device.  The network is the caller's (out of scope); this leg shows the
    post-processing's share of an end-to-end frame and the frames/s the pair reaches, per GPU and over all ranks."""
    import oracle   # only to LOCATE the byte-compiled reference network (an input generator, not a checker here)
    from torch_ekpose_b200 import estimator
    vgg = oracle.reference_module("lib.network.vgg2016")
    torch.manual_seed(0)
    devnull = open(os.devnull, "w")
    old = sys.stdout
    sys.stdout = devnull
    try:
        net = vgg.OpenPose()
    finally:
        sys.stdout = old
        devnull.close()
    net = net.to(dev).eval()
    nb = 32
    rng = np.random.default_rng(5 + rank)
    frames = [rng.integers(0, 255, (368, 432, 3), dtype=np.uint8) for _ in range(nb)]
    out = {"workload": f"configs[4]: {nb} frames of 368x432 per step per GPU -> GPU padding/normalisation -> reference vgg2016 (random init, cuDNN) -> "
                       "post-processing (reference front-end) on the same GPU",
           "model": "lib/network/vgg2016.py OpenPose, unmodified", "params_m": sum(p.numel() for p in net.parameters()) / 1e6}
    for name, dtype in (("fp32", None), ("bf16_autocast", torch.bfloat16)):
        def step():
            with torch.autocast("cuda", dtype=dtype, enabled=dtype is not None):
                return estimator.infer_humans(frames, net, "vgg", dev, frontend="reference")
        for _ in range(2):
            step()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        reps = 4
        t0 = time.perf_counter()
        for _ in range(reps):
            humans = step()
        b.record()
        barrier()
        wall = (time.perf_counter() - t0) / reps
        ms = max(a.elapsed_time(b) / reps, 1000 * wall)
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt[0])
        pp = estimator.last_postprocessor()
        pp.set_timing(True)
        step()
        st, _ = pp.stage_times()
        pp.set_timing(False)
        post = sum(st.values())
        out[name] = {"ms_per_step": ms, "frames_per_s_per_gpu": nb / (ms / 1e3), "frames_per_s_whole_job": world * nb / (ms / 1e3),
                     "postprocess_ms": post, "postprocess_share": post / ms, "humans_last_step": int(sum(len(h) for h in humans))}
    out["note"] = ("random-init heat maps stay below the 0.15 threshold (SURVEY.md 8d), so the post-processing finds no people here: its cost on "
                   "real detections is the c2_*_reference_lean entry (same shapes)")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="skip the configs[2..4] context legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the timed loop's last step to DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # single-process launch asked for N GPUs: re-launch under torchrun as the driver would
        import subprocess
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.abspath(__file__), "--gpus", str(args.gpus),
               "--steps", str(args.steps), "--warmup", str(args.warmup)]
        if args.headline_only:
            cmd.append("--headline-only")
        if args.dump_outputs:
            cmd += ["--dump-outputs", os.path.abspath(args.dump_outputs)]
        raise SystemExit(subprocess.call(cmd))
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
