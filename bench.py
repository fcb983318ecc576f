#!/usr/bin/env python
"""bench.py -- keyframe-pair Jacobian+JtJ evaluations per second (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (libdfk.so)
  python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port, all host threads)
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's results to DIR/*.npy

Workload (BASELINE.json configs[1]): one evaluation = SfmAligner::RunStep over the 4-level pyramid
(640x480 ... 80x60, 408 000 px) of one keyframe/frame pair at code size 32, synthetic data
(deepfactors_b200/synth.py), fp32.  One STEP = `--pairs-per-step` (default 8) such evaluations of DISTINCT
pairs submitted as one persistent launch (8 pairs = 496 MB of inputs > the 126 MB L2, so every step streams its
inputs from HBM); at N > 1 every rank evaluates its own pairs (weak scaling: pairs shard across GPUs with no
data-path collective) and the per-pair normal equations are summed into the window's Hessian buffer with one NCCL
all-reduce per step.  `value` = evaluations of all ranks / max-over-ranks device time.

Keys beyond the base contract: `roofline` (dominant kernel = sfm_step kernel; achieved = algorithmic bytes per
launch / CUDA-event time of the kernel launches in the timed region; peak = MEASURED_PEAKS.json hbm_gbs),
`cpu_baseline` (oracle port, OpenMP, all host cores, bounded sample), `e2e` (same metric through the synchronous
C-ABI call with every input uploaded from pinned host memory and the result read back, each step),
`single_launch` (one pair per launch: the latency-bound regime of the per-factor API).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from

METRIC = "keyframe-pair Jacobian+JtJ evals/sec (640x480, C=32)"
W0, H0, CS, LEVELS = 640, 480, 32, 4
PIXELS = sum((W0 >> l) * (H0 >> l) for l in range(LEVELS))  # 408000
BYTES_PER_PX = 24 + 4 * CS                                  # SURVEY 8(d)
BYTES_PER_EVAL = PIXELS * BYTES_PER_PX                      # 62.02 MB


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="pair8", choices=["pair8", "window200", "ba2k", "c128"],
                    help="pair8 = BASELINE configs[1] (default, the metric's configuration); window200 = configs[2]; ba2k = "
                         "configs[3] (run it with --gpus 8 under torchrun); c128 = configs[4]")
    ap.add_argument("--pairs-per-step", type=int, default=0, help="override the pairs per GPU and step of a 'pairs' config")
    ap.add_argument("--gram", default="auto", choices=["auto", "fp32", "tf32x3"])
    ap.add_argument("--e2e-steps", type=int, default=60)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--code-sigma", type=float, default=0.0,
                    help="std of the latent code used to decode dpt0 (0 = the reference test's zero code, smooth depth; "
                         ">0 adds per-pixel depth noise through the iid synthetic code Jacobian)")
    ap.add_argument("--fused-depth", action="store_true",
                    help="decode dpt0 from prx_orig + code inside the launch (UpdateDepth + RunStep in one pass; "
                         "28+4C algorithmic bytes per pixel instead of 24+4C, and no separate UpdateDepth pass)")
    ap.add_argument("--identity-pose", action="store_true", help="100%% inliers (worst-case work) instead of the ~60%% of the reference test poses")
    ap.add_argument("--no-verify", action="store_true",
                    help="skip the parity check of the TIMED batch against the CPU oracle (outside the timed region)")
    ap.add_argument("--reserve-sms", type=int, default=-1,
                    help="SMs the persistent step kernel leaves free for the concurrent all-reduce of the previous step "
                         "(dfk_set_sm_limit); default: 4 when the job has more than one rank, else 0")
    ap.add_argument("--sustain-seconds", type=float, default=1.2,
                    help="after the K timed steps, repeat the same step back to back for about this long (clocks are sampled "
                         "over both regions); reported as `sustained`")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (per work item: "
                         "JtJ packed upper, Jtr, residual, inliers; the window's block-sparse buffer), for comparing two "
                         "builds on the same seeded inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line).

    The timed region of the default run is tens of milliseconds, shorter than one `nvidia-smi -lms` period, so the
    samples come from NVML directly (nvidia_ml_py), polled from a thread about every millisecond between start()
    and stop(); `nvidia-smi --query-gpu` is only the fallback when NVML cannot be loaded."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        try:
            ids = [int(x) for x in vis.split(",")] if vis else []
            self.index = ids[index] if index < len(ids) else index
        except ValueError:
            self.index = index
        self.samples, self.masks = [], []
        self.max_mhz = None
        self.nvml = self.handle = self.thread = None
        self.running = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _poll_once(self):
        n = self.nvml
        self.samples.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        try:
            fn = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
            self.masks.append(int(fn(self.handle)))
        except Exception:
            pass

    def _loop(self):
        while self.running:
            try:
                self._poll_once()
            except Exception:
                break
            time.sleep(0.001)

    def start(self):
        if self.nvml is None:
            return
        self.running = True
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        if self.nvml is None:
            return self._smi_fallback()
        self.running = False
        if self.thread is not None:
            self.thread.join(timeout=2)
        sm = sorted(self.samples)
        reasons = set()
        for m in self.masks:
            for bit, name in self.REASONS.items():
                if m & bit:
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(reasons),
                "samples": len(sm), "source": "NVML polled during the timed region"}

    def _smi_fallback(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                  str(self.index)], capture_output=True, text=True, timeout=10).stdout.strip()
            f = [x.strip() for x in out.split(",")]
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            reasons = [n for n, v in zip(names, f[2:6]) if v.lower().startswith("active")]
            return {"sm_mhz": float(f[0]), "sm_max_mhz": float(f[1]), "reasons": reasons, "samples": 1,
                    "source": "nvidia-smi one-shot right after the timed region (NVML unavailable)"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}


# ------------------------------------------------------------------------------------------------ CPU arm
def host_cores() -> dict:
    """Host cores this process can really use: the scheduler affinity mask (NOT omp_get_max_threads(): torchrun exports
    OMP_NUM_THREADS=1) capped by the cgroup CPU quota (cpu.max / cfs_quota_us) when one is set."""
    try:
        aff = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        aff = max(1, os.cpu_count() or 1)
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:  # cgroup v2: "<quota|max> <period>"
            q, per = f.read().split()
            if q != "max":
                quota = float(q) / float(per)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                per = float(f.read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    usable = aff if quota is None else max(1, min(aff, int(quota + 0.999)))
    return {"affinity": aff, "cgroup_quota": quota, "usable": usable}


def _cpu_engine(kind):
    """('reference', fn) = the reference's own headers (oracle/_ref, x outer / y inner host loop of ut_sfmaligner.cpp);
    ('port', fn) = the oracle port (row-major).  fn(threads, evals_per_thread) -> wall seconds."""
    from oracle import oracle as orc
    orc.build()
    if kind == "reference":
        from oracle import ref
        if not ref.available():
            return None
        ref.lib()
        return ref
    return orc


def cpu_throughput(kind: str, budget_s: float, code_sigma: float = 0.0, identity_pose: bool = False, sweep=True):
    """CPU arm in THROUGHPUT mode: T threads, each evaluating whole pairs with the reference's single-threaded CPU path
    (no OpenMP, no shared state, nothing spinning) -- what T host cores deliver.  T is swept over {1, 8, 16, 32, 64, all
    usable} in the warm-up and the fastest is timed for ~budget_s seconds.  Returns (record, pair)."""
    from deepfactors_b200 import synth
    eng = _cpu_engine(kind)
    if eng is None:
        kind = "port"
        eng = _cpu_engine("port")
    pair = synth.make_pair(W0, H0, CS, LEVELS, seed=0, code_sigma=code_sigma, identity_pose=identity_pose)
    cores = host_cores()

    def run(threads, evals):
        dt, _ = eng.sfm_throughput(pair.pose0, pair.pose1, pair.levels, threads, evals)
        return dt

    t1 = run(1, 1)  # warm-up + single-thread time of one evaluation
    single = 1.0 / t1
    cand = sorted({c for c in (1, 8, 16, 32, 64, cores["usable"]) if c <= cores["usable"]})
    sweep_res = {1: single}
    best_t, best_v = 1, single
    if sweep:
        for c in cand:
            if c == 1:
                continue
            v = c / run(c, 1)
            sweep_res[c] = v
            if v > best_v:
                best_t, best_v = c, v
    else:
        best_t = cores["usable"]
        best_v = best_t / run(best_t, 1)
    per_round = best_t / best_v  # seconds for one evaluation per thread
    evals = max(1, min(200, int(budget_s / max(per_round, 1e-3))))
    dt = run(best_t, evals)
    value = best_t * evals / dt
    rec = {"value": value, "unit": "evals/s", "cores": best_t, "kind": kind,
           "threads_used": best_t, "host": cores,
           "single_thread": {"value": single, "unit": "evals/s"},
           "thread_sweep_evals_per_s": {str(k): round(v, 2) for k, v in sorted(sweep_res.items())},
           "sample": f"{best_t} threads x {evals} evaluations of one 640x480 4-level C=32 pair ({dt:.1f} s wall), each "
                     "thread running the single-threaded CPU path on its own ("
                     + ("reference headers compiled against oracle/shim, x outer / y inner as ut_sfmaligner.cpp:303-315"
                        if kind == "reference" else "oracle port, fp32, row-major") + ")"}
    return rec, pair


def cpu_baseline(budget_s: float, code_sigma: float = 0.0, identity_pose: bool = False):
    rec, pair = cpu_throughput("port", budget_s, code_sigma, identity_pose)
    # SURVEY 8(d): also the reference's own code, one thread, its test's loop order (ut_sfmaligner.cpp:303-315)
    try:
        eng = _cpu_engine("reference")
        if eng is not None:
            dt, _ = eng.sfm_throughput(pair.pose0, pair.pose1, pair.levels, 1, 1)
            rec["reference_headers_single_thread"] = {"value": 1.0 / dt, "unit": "evals/s", "cores": 1,
                                                      "sample": "1 evaluation through oracle/_ref (the reference's own "
                                                                "dense_sfm.h / warping.h), x outer / y inner"}
    except Exception as e:  # the checker library is optional for this leg
        rec["reference_headers_single_thread"] = {"unavailable": str(e)[:120]}
    return rec, pair


def run_reference_arm(args):
    """`--impl reference`: the reference's own CPU implementation of the path (oracle/_ref: its headers compiled here)
    on all the host threads it can use; one STEP = one evaluation on every thread (a bounded sample of the GPU arm's
    step).  Falls back to the oracle port when oracle/_ref is absent."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from deepfactors_b200 import synth
    kind = "reference"
    eng = _cpu_engine("reference")
    if eng is None:
        kind, eng = "port", _cpu_engine("port")
    pair = synth.make_pair(W0, H0, CS, LEVELS, seed=0, code_sigma=args.code_sigma, identity_pose=args.identity_pose)
    cores = host_cores()

    def run(threads, evals):
        dt, _ = eng.sfm_throughput(pair.pose0, pair.pose1, pair.levels, threads, evals)
        return dt

    single = 1.0 / run(1, 1)
    sweep_res = {1: single}
    best_t, best_v = 1, single
    for c in sorted({c for c in (8, 16, 32, 64, cores["usable"]) if 1 < c <= cores["usable"]}):
        v = c / run(c, 1)  # doubles as the warm-up
        sweep_res[c] = v
        if v > best_v:
            best_t, best_v = c, v
    steps = max(1, args.steps)
    dt = run(best_t, steps)
    val = best_t * steps / dt
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": "evals/s", "n_gpus": args.gpus,
           "steps": steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "single pair 640x480 4-level pyramid, code dim 32 (BASELINE configs[1])",
                      "evals_per_step": best_t,
                      "note": ("reference CPU path = the reference's own headers (dense_sfm.h, warping.h, "
                               "pinhole_camera_impl.h) compiled from /root/reference against the stand-in "
                               "Eigen/Sophus/VisionCore of oracle/shim (those libraries are not installed); host loop of "
                               "tests/ut_sfmaligner.cpp:303-315, one independent single-threaded instance per host thread")
                      if kind == "reference" else "reference CPU path = oracle port of df::DenseSfm (oracle/_ref absent)"},
           "cpu_baseline": {"value": val, "unit": "evals/s", "cores": best_t, "kind": kind, "threads_used": best_t,
                            "host": cores, "single_thread": {"value": single, "unit": "evals/s"},
                            "thread_sweep_evals_per_s": {str(k): round(v, 2) for k, v in sorted(sweep_res.items())},
                            "sample": f"{steps} steps x {best_t} threads, one evaluation per thread and step"},
           "e2e": {"value": val, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------------ e2e
def run_e2e(args, al, base, host_levels, cs, dev, world, dist):
    """The same metric through the reference-facing C-ABI call with HOST buffers: dfk_sfm_stream_submit / _wait
    (include/dfk.h).  Every step uploads ALL inputs of one evaluation (4 levels x img0, img1, dpt0, prx_jac, grad1) from
    pinned host memory, evaluates them and brings the 4 result records back to host memory; up to 3 submissions are in
    flight, so the upload of evaluation k+1 overlaps the kernels of evaluation k (one synchronisation per wait)."""
    import ctypes as C

    import numpy as np
    import torch

    from deepfactors_b200 import _lib
    from deepfactors_b200._lib import DfkCamera, DfkImage, DfkSfmWorkItem

    lib = _lib.lib()
    rec_floats = _lib.record_floats(cs)
    in_keys = ["img0", "img1", "prx0_jac", "grad1"] + (["prx_orig"] if args.fused_depth else ["dpt0"])
    pinned = [{k: torch.from_numpy(np.ascontiguousarray(hl[k], dtype=np.float32)).pin_memory() for k in in_keys}
              for hl in host_levels]
    h2d = sum(int(t.numel()) * 4 for lv in pinned for t in lv.values())
    d2h = LEVELS * rec_floats * 4

    def himg(t, k=1):
        H = t.shape[0]
        W = t.shape[1] if t.dim() == 2 else t.shape[1]
        return DfkImage(C.c_void_p(t.data_ptr()), t.stride(0) * 4, W, H)

    arr = (DfkSfmWorkItem * LEVELS)()
    code_keep = np.ascontiguousarray(base.code, dtype=np.float32)
    for l, (L, pl) in enumerate(zip(base.levels, pinned)):
        w = arr[l]
        w.pose0 = (C.c_float * 7)(*np.asarray(base.pose0, dtype=np.float32).tolist())
        w.pose1 = (C.c_float * 7)(*np.asarray(base.pose1, dtype=np.float32).tolist())
        w.cam = DfkCamera(L.cam.fx, L.cam.fy, L.cam.u0, L.cam.v0, L.cam.width, L.cam.height)
        w.img0, w.img1, w.prx0_jac, w.grad1 = himg(pl["img0"]), himg(pl["img1"]), himg(pl["prx0_jac"]), himg(pl["grad1"])
        if args.fused_depth:
            w.prx_orig = himg(pl["prx_orig"])
            w.code = code_keep.ctypes.data_as(C.POINTER(C.c_float))
        else:
            w.dpt0 = himg(pl["dpt0"])
    depth = 3
    stream = C.c_void_p()
    al._hd.use_torch_stream()
    _lib.check(al.handle, lib.dfk_sfm_stream_create(al.handle, cs, LEVELS, h2d + (1 << 20), depth, C.byref(stream)))
    out = np.zeros((LEVELS, rec_floats), dtype=np.float32)
    outp = out.ctypes.data_as(C.POINTER(C.c_float))
    tk = C.c_uint64(0)

    def run(n):
        waited = 0
        for k in range(n):
            if k - waited >= depth:
                _lib.check(al.handle, lib.dfk_sfm_stream_wait(al.handle, stream, C.c_uint64(first + waited), outp))
                waited += 1
            _lib.check(al.handle, lib.dfk_sfm_stream_submit(al.handle, stream, arr, LEVELS, C.byref(tk)))
        while waited < n:
            _lib.check(al.handle, lib.dfk_sfm_stream_wait(al.handle, stream, C.c_uint64(first + waited), outp))
            waited += 1

    first = 0
    run(3)              # warm-up (also sizes the handle's scratch)
    first += 3
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    n = max(1, args.e2e_steps)
    t0 = time.perf_counter()
    run(n)
    e2e_dt = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_dt, op=dist.ReduceOp.MAX)
    value = world * n / float(e2e_dt.item())
    # the records that came back are the evaluation of the base pair: a cheap sanity check against a device-resident run
    inl = int(out[0][-1:].view(np.uint32)[0])
    lib.dfk_sfm_stream_destroy(al.handle, stream)
    return {"value": value, "unit": "evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": n,
            "gb_per_s_h2d": value / max(world, 1) * h2d / 1e9, "pipeline_depth": depth, "level0_inliers_returned": inl,
            "note": "per step: dfk_sfm_stream_submit with HOST (pinned) image views of one evaluation -- every level's "
                    "img0/img1/dpt0/prx_jac/grad1 uploaded on a copy stream, one batched launch for the 4 levels, the 4 "
                    "result records downloaded -- and dfk_sfm_stream_wait; 3 submissions in flight"}


# ------------------------------------------------------------------------------------------------ GPU arm
CONFIGS = {
    # BASELINE.json configs[1], the metric's own configuration: 8 distinct pairs per GPU and step
    "pair8": dict(kind="pairs", code=32, pairs_per_gpu=8,
                  workload="single pair 640x480 4-level pyramid, code dim 32 (BASELINE configs[1]); {P} distinct pairs per "
                           "GPU and step in one persistent launch"),
    # configs[2]: one Gauss-Newton linearisation of a 50-keyframe window with 200 co-visibility pairs on one GPU
    "window200": dict(kind="window", code=32, keyframes=50, pairs=200,
                      workload="50-keyframe window, 200 co-visibility pairs (ring + random, seed 2), code dim 32, 640x480 "
                               "4-level pyramids (BASELINE configs[2]); one step = one linearisation of the window"),
    # configs[3]: global BA, pairs sharded over the GPUs, one all-reduce of the block-sparse Hessian per step
    "ba2k": dict(kind="window", code=32, keyframes=200, pairs=2000,
                 workload="200-keyframe global BA, 2000 pairs sharded over the GPUs, code dim 32, 640x480 4-level pyramids "
                          "(BASELINE configs[3]); one step = one linearisation + the all-reduce of the block-sparse Hessian"),
    # configs[4]: the code size the reference declares but cannot launch (cu_sfmaligner.cpp:170-173,210-211)
    "c128": dict(kind="pairs", code=128, pairs_per_gpu=2,
                 workload="single pair 640x480 4-level pyramid, code dim 128 (BASELINE configs[4]); {P} distinct pairs per "
                          "GPU and step"),
}


def window_pairs(num_kf: int, num_pairs: int, seed: int = 2):
    """SURVEY 8d(iii): ring neighbours first ((k, k+1), (k, k+2), ...), then random co-visibility pairs."""
    import numpy as np
    pairs, seen = [], set()
    d = 1
    while len(pairs) < min(num_pairs, num_kf * 5) and d <= 5:
        for k in range(num_kf):
            if len(pairs) >= num_pairs:
                break
            pr = (k, (k + d) % num_kf)
            if pr not in seen:
                seen.add(pr)
                pairs.append(pr)
        d += 1
    rng = np.random.default_rng(seed)
    while len(pairs) < num_pairs:
        a, b = int(rng.integers(num_kf)), int(rng.integers(num_kf))
        if a != b and (a, b) not in seen:
            seen.add((a, b))
            pairs.append((a, b))
    return pairs


DUMP_BYTES = 64 << 20


def dump_outputs(path, cs, records, window):
    """--dump-outputs: the result records of one step and the window buffer they were assembled into, as float32 / float64
    .npy files.  Above DUMP_BYTES in all, every array is flattened and keeps the same share of its elements, at positions
    drawn from a fixed seed, so two runs of one configuration store the same positions."""
    import numpy as np

    from deepfactors_b200 import factors
    n, nh, _ = factors.record_layout(cs)
    arrays = {"JtJ": records[:, :nh], "Jtr": records[:, nh:nh + n], "residual": records[:, nh + n],
              "inliers": np.ascontiguousarray(records[:, nh + n + 1]).view(np.uint32).astype(np.float64),
              "window": window}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = a.size * (DUMP_BYTES - (1 << 16)) // total   # headroom for the .npy headers
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a))


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import ctypes as C

    import numpy as np
    import torch
    import torch.distributed as dist

    from deepfactors_b200 import _lib, synth
    from deepfactors_b200.aligners import SfmAligner, Window

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        # the per-step collective is a few hundred KB: two channels are plenty, and a small NCCL grid fits into the SMs the step
        # kernel leaves free (see --reserve-sms)
        os.environ.setdefault("NCCL_MAX_NCHANNELS", "2")
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    cfg = CONFIGS[args.config]
    cs = cfg["code"]
    if cfg["kind"] == "pairs" and args.pairs_per_step:
        cfg = dict(cfg, pairs_per_gpu=args.pairs_per_step)

    # ---- synthetic data resident in HBM ----------------------------------------------------------------------------
    base = synth.make_pair(W0, H0, cs, LEVELS, seed=rank if cfg["kind"] == "pairs" else 0, code_sigma=args.code_sigma,
                           identity_pose=args.identity_pose)
    host_levels = []
    for L in base.levels:
        host_levels.append(dict(img0=L.img0, img1=L.img1, dpt0=L.dpt0, prx0_jac=L.prx_jac, grad1=L.grad1))
        if args.fused_depth:
            host_levels[-1]["prx_orig"] = L.prx_orig
    base_dev = [{k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in hl.items()} for hl in host_levels]

    def variant(l, q):
        """inputs of level l, variation q (q = 0: the host-generated base): distinct contents per pair / keyframe made on
        the device -- the code Jacobian rolled, img0 scaled.  bench_host_variant() repeats it on the host for --verify."""
        d = dict(base_dev[l])
        if q > 0:
            d["prx0_jac"] = torch.roll(d["prx0_jac"], shifts=(3 * q, 5 * q), dims=(0, 1)).contiguous()
            d["img0"] = (d["img0"] * (1.0 - 0.01 * (q % 50))).contiguous()
            # every variation owns ALL of its buffers (same contents for img1 / grad1 / dpt0, different memory): pairs that
            # shared them would turn the bilinear gathers of 7 of 8 pairs into L2 hits (measured: -13 % kernel time)
            for k in ("img1", "grad1", "dpt0", "prx_orig"):
                if k in d:
                    d[k] = d[k].clone()
        d["valid0"] = torch.zeros_like(d["img0"])
        return d

    def host_variant(l, q):
        L = base.levels[l]
        jac = np.roll(L.prx_jac, shift=(3 * q, 5 * q), axis=(0, 1)) if q > 0 else L.prx_jac
        img0 = (L.img0 * np.float32(1.0 - 0.01 * (q % 50))).astype(np.float32) if q > 0 else L.img0
        return np.ascontiguousarray(jac), img0

    al = SfmAligner(cs, gram_mode=args.gram)
    reserve_sms = args.reserve_sms if args.reserve_sms >= 0 else (4 if world > 1 else 0)
    if reserve_sms > 0:
        al.SetSmLimit(torch.cuda.get_device_properties(dev).multi_processor_count - reserve_sms)
    items, item_pair, item_sizes, item_src = [], [], [], []   # item_src: (variation of img0/jac side, level) for --verify
    if cfg["kind"] == "pairs":
        P = cfg["pairs_per_gpu"]            # pairs of THIS rank; the window of all ranks has world * P pairs
        num_kf = 2 * P * world              # every pair brings its own keyframe and frame
        all_pairs = [(2 * p, 2 * p + 1) for p in range(P * world)]
        for p in range(P):
            for l, L in enumerate(base.levels):
                d = variant(l, p)
                items.append(dict(pose0=base.pose0, pose1=base.pose1, cam=L.cam, img0=d["img0"], img1=d["img1"],
                                  dpt0=d["dpt0"], valid0=d["valid0"], prx0_jac=d["prx0_jac"], grad1=d["grad1"]))
                if args.fused_depth:
                    items[-1].update(prx_orig=d["prx_orig"], code=base.code)
                item_pair.append(rank * P + p)
                item_sizes.append((L.width, L.height))
                item_src.append((p, l))
        scaling = "weak"
    else:
        num_kf = cfg["keyframes"]
        all_pairs = window_pairs(num_kf, cfg["pairs"])
        lo, hi = (len(all_pairs) * rank) // world, (len(all_pairs) * (rank + 1)) // world   # factors.shard_pairs
        kfs = {}
        for p in range(lo, hi):
            for k in all_pairs[p]:
                if k not in kfs:
                    kfs[k] = [variant(l, k) for l in range(LEVELS)]   # keyframe k: its own buffers at every level
        for p in range(lo, hi):
            k0, k1 = all_pairs[p]
            for l, L in enumerate(base.levels):
                a, b = kfs[k0][l], kfs[k1][l]
                items.append(dict(pose0=base.pose0, pose1=base.pose1, cam=L.cam, img0=a["img0"], img1=b["img1"],
                                  dpt0=a["dpt0"], valid0=a["valid0"], prx0_jac=a["prx0_jac"], grad1=b["grad1"]))
                if args.fused_depth:
                    items[-1].update(prx_orig=a["prx_orig"], code=base.code)
                item_pair.append(p)
                item_sizes.append((L.width, L.height))
                item_src.append((k0, l))
        P = hi - lo
        scaling = "strong"
    work = al.make_work_items(items)
    rec_floats = _lib.record_floats(cs)
    n_items = len(items)
    records = torch.zeros((n_items, rec_floats), dtype=torch.float32, device=dev)
    # the window's block-sparse normal equations: every rank assembles ITS pairs into the layout of the WHOLE window, one
    # all-reduce (sum) per step joins the ranks; two buffers so the collective of step i overlaps step i+1
    win = Window(al, num_kf, all_pairs, item_pair, item_sizes)
    wbuf = [torch.zeros(win.floats, dtype=torch.float32, device=dev) for _ in range(2)]
    pending = [None, None]
    step_no = [0]

    def step():
        i = step_no[0] & 1
        if pending[i] is not None:
            pending[i].wait()           # the collective that last used this buffer (two steps ago): stream-side wait only
            pending[i] = None
        al.RunStepBatch(work, records)
        win.assemble(records, wbuf[i])
        if world > 1:
            pending[i] = dist.all_reduce(wbuf[i], async_op=True)
        step_no[0] += 1

    def drain_comm():
        for i in range(2):
            if pending[i] is not None:
                pending[i].wait()
                pending[i] = None

    lib = _lib.lib()

    def read_profile():
        ms, n, tot = C.c_double(0), C.c_uint64(0), C.c_uint64(0)
        _lib.check(al.handle, lib.dfk_get_profile(al.handle, C.byref(ms), C.byref(n), C.byref(tot)))
        return ms.value, n.value, tot.value

    for _ in range(max(3, args.warmup)):
        step()
    drain_comm()
    torch.cuda.synchronize()
    read_profile()
    _lib.check(al.handle, lib.dfk_set_profiling(al.handle, 1))

    def aligned_start():
        """barrier + synchronize (the contract), then one tiny all-reduce ON the launch stream right before the start event:
        the host-side barrier releases the ranks up to a millisecond apart (8 Python processes), and a rank that starts
        early would wait that skew out inside its first collective and count it; the in-stream collective completes on all
        ranks within microseconds, so every rank's clock starts at the same point of the job"""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if world > 1:
            dist.all_reduce(align_buf)
    align_buf = torch.zeros(1, device=dev)

    aligned_start()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # Lead-in: the W warm-up steps are issued again BEHIND the barrier + synchronize and run straight into the timed steps
    # (the start event is recorded in-stream between them).  Each step overlaps the previous step's collective and the
    # host runs ahead of the device; coming out of a synchronize that pipeline takes a few steps to fill (0.5 - 4 ms at
    # N = 2 .. 8), which a 20-step region would charge to the steady-state rate the metric is about.  The K timed steps,
    # their collectives and the final drain are all inside [e0, e1].
    lead_in = max(3, args.warmup) if world == 1 else max(8, args.warmup)   # ranks couple through collectives two steps deep
    for _ in range(lead_in):
        step()
    e0.record()
    for _ in range(args.steps):
        step()
    drain_comm()                      # the last steps' all-reduces belong to the timed region
    e1.record()
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, cs, records.cpu().numpy(), wbuf[(step_no[0] - 1) & 1].cpu().numpy())
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    kern_ms, kern_n, launches = read_profile()   # covers the lead-in steps too: scale the counts to the K timed steps
    launches = launches * args.steps / (lead_in + args.steps)
    kern_ms, kern_n = kern_ms * args.steps / (lead_in + args.steps), kern_n * args.steps / (lead_in + args.steps)
    pairs_all_ranks = torch.tensor([float(P)], device=dev)
    if world > 1:
        dist.all_reduce(pairs_all_ranks)
    evals_per_step = float(pairs_all_ranks.item())
    value = evals_per_step * args.steps / (total_ms * 1e-3)

    # ---- sustained region: the same step, back to back, for >= --sustain-seconds (a few-ms region is a sanity check, not
    # a headline; this one is long enough for the clock / power state to settle and for NVML to see it)
    sustained = None
    if args.sustain_seconds > 0:
        n_sus = max(args.steps, int(args.sustain_seconds * 1e3 / max(total_ms / args.steps, 1e-3)) + 1)
        aligned_start()
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        q0.record()
        for _ in range(n_sus):
            step()
        drain_comm()
        q1.record()
        torch.cuda.synchronize()
        sms = torch.tensor([q0.elapsed_time(q1)], device=dev)
        if world > 1:
            dist.all_reduce(sms, op=dist.ReduceOp.MAX)
        sus_ms = float(sms.item())
        k2_ms, k2_n, _ = read_profile()
        sustained = {"steps": n_sus, "seconds": sus_ms * 1e-3, "value": evals_per_step * n_sus / (sus_ms * 1e-3),
                     "unit": "evals/s", "ms_per_step": sus_ms / n_sus,
                     "kernel_avg_launch_ms": (k2_ms / k2_n) if k2_n else None}
    clocks = sampler.stop() if rank == 0 else None
    _lib.check(al.handle, lib.dfk_set_profiling(al.handle, 0))

    # ---- parity of the TIMED batch (outside the timed regions): records of the first and the last pair of this rank, all
    # levels, against the CPU oracle on the same inputs; and the window buffer against the host mirror of the assembly
    parity = None
    if rank == 0 and not args.no_verify:
        from deepfactors_b200 import factors
        from oracle import oracle as orc
        orc.build()
        al.RunStepBatch(work, records)          # a private evaluation: at N > 1 the window buffers hold reduced sums
        chk = win.assemble(records)
        torch.cuda.synchronize()
        recs_host = records.cpu().numpy()
        NP = 12 + cs
        NH = NP * (NP + 1) // 2
        worst_h, worst_g, inl_ok, checked, border_cases = 0.0, 0.0, True, 0, 0
        prm = orc.default_params()
        first, last = 0, n_items - LEVELS
        for it0 in sorted({first, last}):
            for l in range(LEVELS):
                i = it0 + l
                q, lv = item_src[i]
                L = base.levels[lv]
                jac, img0 = host_variant(lv, q)
                dpt0 = L.dpt0
                if args.fused_depth:
                    dpt0 = orc.update_depth(base.code, L.prx_orig, jac, 2.0)
                o = orc.sfm_run_step(base.pose0, base.pose1, L.cam, img0, L.img1, dpt0, None, jac, L.grad1, prm,
                                     precision="f64")
                of = orc.sfm_run_step(base.pose0, base.pose1, L.cam, img0, L.img1, dpt0, None, jac, L.grad1, prm,
                                      precision="f32")
                r = recs_host[i]
                inl = int(r[NH + NP + 1:NH + NP + 2].view(np.uint32)[0])
                # inlier set: bit-exact against the fp32 CPU path (what the reference's own GPU-vs-CPU test demands,
                # ut_sfmaligner.cpp:320).  fp64 can disagree with fp32 about pixels exactly on the border line (identity
                # poses): then the sums are compared with the fp32 flavour, at its own accumulation error.
                inl_ok = inl_ok and (inl == of.inliers)
                ref_o, scale = (o, 1.0) if o.inliers == of.inliers else (of, 2.0)
                border_cases += int(o.inliers != of.inliers)
                hmax = float(np.abs(ref_o.JtJ).max()) or 1.0
                worst_h = max(worst_h, float(np.abs(r[:NH] - ref_o.JtJ).max()) / hmax / scale)
                worst_g = max(worst_g, float(np.abs(r[NH:NH + NP] - ref_o.Jtr).max()) /
                              (float(np.abs(ref_o.Jtr).max()) or 1.0) / scale)
                checked += 1
        Hh, gh, rh, ih = factors.unpack_records(recs_host, cs)
        want = win.layout.pack(item_pair, Hh, gh, rh, ih, item_sizes)
        got = chk.cpu().numpy()
        win_err = float(np.abs(got - want).max() / (np.abs(want).max() or 1.0))
        tol_h = 2e-5 if cs <= 32 else 4e-5
        parity = {"parity_checked": True, "records_checked": checked, "inliers_exact": bool(inl_ok),
                  "max_rel_err_JtJ_vs_f64": worst_h, "max_rel_err_Jtr_vs_f64": worst_g,
                  "tolerance": {"JtJ": tol_h, "Jtr": 1e-4, "window": 2e-6},
                  "window_buffer_max_rel_err_vs_host_mirror": win_err,
                  "ok": bool(inl_ok and worst_h <= tol_h and worst_g <= 1e-4 and win_err <= 2e-6),
                  "records_compared_with_fp32_flavour": border_cases,
                  "what": "first and last pair of the timed batch, all levels: inliers vs the fp32 CPU path (exact), sums vs "
                          "oracle fp64 (vs fp32 at twice the tolerance where fp64 and fp32 disagree on border pixels); the "
                          "assembled block-sparse window vs factors.WindowBlocks.pack on the same records"}

    # ---- single pair per launch (latency-bound regime: what PhotometricFactor::linearize pays per factor) ---------------
    single = None
    if cfg["kind"] == "pairs":
        works1 = [al.make_work_items(items[p * LEVELS:(p + 1) * LEVELS]) for p in range(P)]
        recs1 = torch.empty((LEVELS, rec_floats), dtype=torch.float32, device=dev)
        for p in range(P):
            al.RunStepBatch(works1[p], recs1)
        torch.cuda.synchronize()
        n1 = max(50, 4 * args.steps)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for i in range(n1):
            al.RunStepBatch(works1[i % P], recs1)
        s1.record()
        torch.cuda.synchronize()
        single_ms = s0.elapsed_time(s1) / n1
        single = {"pairs_per_launch": 1, "value": 1e3 / single_ms, "unit": "evals/s", "ms_per_eval": single_ms,
                  "frac_of_hbm_roofline": None}

    # ---- e2e: the same metric through the C-ABI streaming call with HOST buffers ---------------------------------------
    e2e = run_e2e(args, al, base, host_levels, cs, dev, world, dist)

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak = float(json.load(open(peaks_path))["hbm_gbs"])
            peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
        else:
            peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        bytes_per_px = 24 + 4 * cs + (4 if args.fused_depth else 0)   # SURVEY 8(d)
        bytes_per_eval = PIXELS * bytes_per_px
        bytes_per_launch = P * bytes_per_eval
        traffic = None  # dram__bytes_read+write of one step-kernel launch, from the committed ncu --set full capture
        tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tpath) and args.config == "pair8" and P == 8 and args.gram in ("auto", "tf32x3") and not args.fused_depth:
            traffic = json.load(open(tpath))["traffic_bytes_per_launch"]
        kern_avg_ms = kern_ms / max(kern_n, 1)
        achieved = bytes_per_launch / (kern_avg_ms * 1e-3) / 1e9 if kern_n else None
        if single is not None:
            single["frac_of_hbm_roofline"] = (bytes_per_eval / (single["ms_per_eval"] * 1e-3) / 1e9) / peak
        cpu = None
        if not args.no_cpu_baseline and world == 1 and cs == 32:
            cpu, _ = cpu_baseline(args.cpu_seconds, args.code_sigma, args.identity_pose)
        out = {
            "metric": METRIC if cs == 32 else METRIC.replace("C=32", f"C={cs}"), "value": value, "unit": "evals/s",
            "n_gpus": n_gpus, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"name": args.config, "workload": cfg["workload"].format(P=P),
                       "evals_per_step_per_gpu": P, "evals_per_step": evals_per_step, "pixels_per_eval": PIXELS,
                       "algorithmic_bytes_per_eval": bytes_per_eval, "gram": args.gram, "code_size": cs,
                       "fused_depth_decode": bool(args.fused_depth),
                       "poses": "identity (100% inliers)" if args.identity_pose else
                                "tests/ut_sfmaligner.cpp:254-264 (~60% inliers)",
                       "code_sigma": args.code_sigma,
                       "window": {"keyframes": num_kf, "pairs": len(all_pairs), "block_sparse_floats": win.floats,
                                  "block_sparse_bytes": 4 * win.floats},
                       "l2": f"inputs larger than L2: each step streams {P * bytes_per_eval / 1e6:.0f} MB of pair data per GPU "
                             "(> 126 MB L2)" if P * bytes_per_eval > 126e6 else
                             f"{P * bytes_per_eval / 1e6:.0f} MB of pair data per step and GPU",
                       "parallelism": f"pairs sharded over {n_gpus} GPU(s); every step assembles the window's block-sparse "
                                      "normal equations on the device" + (
                           "; ONE NCCL all-reduce of that buffer per step, asynchronous, overlapped with the next step's "
                           f"launch; the step kernel's grid leaves {reserve_sms} SMs to that collective (dfk_set_sm_limit)"
                           if world > 1 else ""),
                       "reserved_sms": reserve_sms,
                       "timing": f"barrier + synchronize, {lead_in} untimed lead-in steps, start event in-stream, EXACTLY "
                                 f"{args.steps} timed steps + the drain of their collectives, stop event, synchronize + "
                                 "barrier; max over ranks of the per-rank event time"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": traffic,
                         "kernel": "sfm_step kernel (per-tile warp + Gram)", "launches_timed": int(round(kern_n)),
                         "avg_launch_ms": kern_avg_ms, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": bytes_per_launch},
            "cpu_baseline": cpu,
            "e2e": e2e,
            "single_launch": single,
            "sustained": sustained,
            "parity": parity,
            "gpu_launches": int(round(launches)),
            "clocks": clocks,
        }
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
