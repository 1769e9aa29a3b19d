#!/usr/bin/env python
"""bench.py -- loop-closure registrations/sec on 100k-point KITTI-shaped pairs (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port + reference nanoflann)
    torchrun ... bench.py --gpus N ...                       # one rank per GPU, weak scaling

Headline (configs[1]): one "step" = LoopClosure::icpAlignment (fast_lio_sam_qn/src/loop_closure.cpp:110-136: two index
builds, two covariance passes, align, fitness) over 256 synthetic 100k x 100k pairs per rank, issued as 16 jobs of 16 pairs
to the C ABI's batch driver (b200reg_batch_*, three engine contexts on C++ host threads).  The jobs rotate over 4 DISTINCT
sub-batches (64 distinct pairs, 205 MB of raw points per rank -- more than the 126 MB L2), nothing is replaced or skipped.
Prints ONE JSON line (rank 0):

  value    : pairs/s with the raw xyz already resident in HBM when the timed region starts
  e2e      : pairs/s through the same C-ABI calls from PINNED HOST buffers (H2D of every cloud of every job and D2H of
             the result records inside the timed region)
  roofline : dominant kernel family, algorithmic bytes (SURVEY.md §8(d)) / CUDA-event time on the launching stream,
             against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline: the CPU oracle (restated Nano-GICP + the reference's own nanoflann from oracle/_ref), bounded sample
  parity   : the GPU transforms of the sampled pairs against the CPU oracle's (1e-4 rad / 1e-3 m, counters equal,
             first-linearize correspondences bit-exact); a miss aborts the run
  latency  : ms per single pair through one C-ABI call on an idle GPU (the reference's published "ms per ICP" view)
  secondary: the other BASELINE configs measured in the same run: configs[2] full loop closure (Quatro + Nano-GICP) on
             0.3 m-voxelised and on RAW 100k scans, configs[4] the 2761-keyframe KITTI-05-shaped sequence through
             loopTimerFunc's steps, and for N > 1 configs[3] the 512-pair batch sharded over the ranks with one
             NCCL all-gather of the result records per batch (b200reg_allgather_results)
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "fast-lio-sam-qn_b200"))

import numpy as np  # noqa: E402

METRIC = "loop_closure_registrations_per_sec_100k_pt_pairs"
UNIT = "pairs/s"
N_POINTS = 100000
JOB_PAIRS = 16        # pairs per b200reg_batch job
DISTINCT_JOBS = 4     # distinct sub-batches the jobs rotate over (4 x 16 pairs x 3.2 MB = 205 MB > L2)
JOBS_PER_STEP = 16    # 256 pairs per step per rank
ROT_TOL, TRANS_TOL = 1e-4, 1e-3


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--points", type=int, default=N_POINTS)
    ap.add_argument("--depth", type=int, default=int(os.environ.get("B200REG_PIPE_DEPTH", "3")),
                    help="engine contexts of the batch driver.  Measured on this workload (value / e2e pairs/s, 20 steps): 2: 4420 / 3811; "
                         "3: 4639 / 4145, 4641 / 4144, 4591 / 4107 (stable); 4: 3856 / 4290 (four contexts over four rotating sub-batches "
                         "fall into lockstep); 5: 4653 / 4383, 4724 / 4372, but also 4066 / 4395 -- more contexts hide more of the uploads "
                         "yet can phase-lock on the device-resident arm, so the default stays at the stable 3")
    ap.add_argument("--depth-e2e", type=int, default=int(os.environ.get("B200REG_PIPE_DEPTH_E2E", "3")),
                    help="engine contexts of the batch driver of the from-host arm (default: the same driver as the device-resident arm). "
                         "It has uploads to hide and rises steadily with the depth (3811 / 4145 / 4290 / 4383 pairs/s at 2 / 3 / 4 / 5; 4420-4434 "
                         "measured at 5 over ~30 runs), but ONE of those runs ended in a CUDA 'illegal memory access' that could not be "
                         "reproduced or explained (profiles/README.md), so the default stays with the configuration that has never failed")
    ap.add_argument("--depth-lc", type=int, default=3,
                    help="engine contexts of the batch driver of the loop-closure secondaries (default: the headline's driver; the coarse "
                         "stage has latency-bound kernels and gains from more contexts in flight -- 4613 / 4745 / 4810 / 4870 pairs/s on the "
                         "voxelised workload at 3 / 5 / 6 / 8 -- but see --depth-e2e for why the defaults stay at 3)")
    ap.add_argument("--secondary", default="all", help="comma list of secondary workloads: voxel,raw,sequence,batch512 | all | none")
    ap.add_argument("--keyframes", type=int, default=2761, help="sequence workload: keyframes generated (KITTI 05: 2761)")
    ap.add_argument("--matching", default="optimized", choices=["optimized", "advanced"])
    ap.add_argument("--cpu-sample-pairs", type=int, default=6)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the result records of the headline's last timed step to DIR/<field>.npy "
                         "(float32 / float64), so that two builds can be compared output for output on the same inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 arm")
    return args


# ---------------------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------------------
def gen_pairs(seeds, n_points, mode="gicp", voxel=None, threads=None):
    """synth.make_pair for every seed (the generator runs OpenMP inside; a few Python threads keep the cores busy).
    A seed whose procedural scene cannot return n_points echoes (the virtual sensor sits inside a building: one in a few
    hundred) is replaced by seed + 100000, deterministically -- an input-generation matter, not a registration one."""
    from b200reg import synth

    def one(s):
        for k in range(4):
            try:
                return synth.make_pair(s + 100000 * k, n_points, n_points, mode=mode, voxel=voxel)
            except RuntimeError:
                continue
        raise RuntimeError("no usable synthetic scene for seed %d" % s)
    threads = threads or max(1, min(16, (os.cpu_count() or 8) // 8))
    with ThreadPoolExecutor(threads) as ex:
        return list(ex.map(one, seeds))


def primary_seeds(rank=0):
    """SURVEY §8(d): config 2 uses seeds 1000...  Weak scaling fixes the per-GPU work, so EVERY rank registers the same pool
    of 64 pairs (each rank starts the rotation at its own sub-batch); synthetic pools differ in cost -- the pool 1064..1127
    holds the 32-iteration seed 1104 and is 12 % heavier (profiles/r02/n2_diag.txt) -- and rank-distinct pools would measure
    that difference, not the system.  They are measured too: `secondary.rank_distinct_pools` (N>1)."""
    return [1000 + i for i in range(JOB_PAIRS * DISTINCT_JOBS)]


def rank_distinct_seeds(rank):
    n = JOB_PAIRS * DISTINCT_JOBS
    return [1000 + rank * n + i for i in range(n)]


def primary_config(args):
    """The workload description -- identical in the b200 and the reference arm."""
    return {"workload": "configs[1]: Nano-GICP %dk-pt KITTI-shaped scan pairs (LoopClosure::icpAlignment: 2 index builds + 2 kNN-15 "
                        "covariance passes + LM align + fitness)" % (args.points // 1000),
            "points_per_cloud": args.points, "pairs_per_step_per_gpu": JOB_PAIRS * JOBS_PER_STEP,
            "distinct_pairs_per_gpu": JOB_PAIRS * DISTINCT_JOBS,
            "seeds": "1000 + i, i < 64, the same pool on every rank (no pair replaced or skipped); rank r starts its rotation at sub-batch r",
            "l2": "the jobs of a step rotate over 4 distinct 16-pair sub-batches: %.0f MB of raw points per rank (> 126 MB L2); "
                  "every job rebuilds all derived data from the raw xyz" % (2 * JOB_PAIRS * DISTINCT_JOBS * args.points * 16 / 1e6)}


class Arena:
    """Pinned-host and device copies of a list of pairs, grouped into jobs of `per_job` pairs."""

    def __init__(self, pairs, per_job):
        import torch
        rebind_cpus()
        self.pairs = pairs
        self.hs = [torch.from_numpy(np.ascontiguousarray(p[0])).pin_memory() for p in pairs]
        self.hd = [torch.from_numpy(np.ascontiguousarray(p[1])).pin_memory() for p in pairs]
        self.ds = [t.cuda(non_blocking=True) for t in self.hs]
        self.dd = [t.cuda(non_blocking=True) for t in self.hd]
        torch.cuda.synchronize()
        self.stride = self.hs[0].shape[1] * 4
        self.jobs = [list(range(i, min(i + per_job, len(pairs)))) for i in range(0, len(pairs), per_job)]

    def job(self, j, on_device):
        idx = self.jobs[j % len(self.jobs)]
        s = self.ds if on_device else self.hs
        d = self.dd if on_device else self.hd
        return ([s[i].data_ptr() for i in idx], [s[i].shape[0] for i in idx], [d[i].data_ptr() for i in idx],
                [d[i].shape[0] for i in idx], self.stride, int(on_device))

    def h2d_bytes(self, j):
        return sum(self.hs[i].numel() * 4 + self.hd[i].numel() * 4 for i in self.jobs[j % len(self.jobs)])


# ---------------------------------------------------------------------------------------------------------------------
# host / clocks
# ---------------------------------------------------------------------------------------------------------------------
_ALL_CPUS = None
_NEAR_CPUS = None


def bind_near_gpu(dev):
    """Run this rank's host threads (and so first-touch its pinned buffers) on the CPUs local to its GPU's PCIe root --
    what `numactl --cpunodebind` does for a production rank.  Returns the cpulist string, None if the topology is not exposed."""
    global _ALL_CPUS, _NEAR_CPUS
    if os.environ.get("B200REG_BENCH_NO_AFFINITY"):
        return None
    try:
        import torch
        p = torch.cuda.get_device_properties(dev)
        bus = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bus) as f:
            txt = f.read().strip()
        cpus = set()
        for part in txt.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if len(cpus) < 16:  # a cpuset that leaves only a few local CPUs: the remote socket is the better place
            return None
        _ALL_CPUS = os.sched_getaffinity(0)
        _NEAR_CPUS = cpus
        os.sched_setaffinity(0, cpus)
        return txt
    except (OSError, ValueError, AttributeError, RuntimeError):
        return None


def unbind_cpus():
    """The CPU baselines use every core of the box."""
    if _ALL_CPUS:
        os.sched_setaffinity(0, _ALL_CPUS)


def rebind_cpus():
    """Back next to the GPU after a CPU baseline (the batch driver's worker threads never left)."""
    if _NEAR_CPUS:
        os.sched_setaffinity(0, _NEAR_CPUS)


def cpu_info():
    model = "unknown"
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    model = line.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    return model, os.cpu_count()


def calibrate_threads(orc, fn, pair):
    """Pick the OpenMP thread count that makes the CPU path FASTEST on this host, best of 3 runs per candidate (all
    logical CPUs is not always it: on the 128-thread GPU-box Xeon the guided-schedule loops are slowest at 128)."""
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cands = sorted({max(1, ncpu >> k) for k in range(0, 4)}, reverse=True)
    best, best_t = cands[0], float("inf")
    src, dst = pair[0], pair[1]
    for n in cands:
        orc.lib().orc_set_num_threads(n)
        fn(src[:20000], dst[:20000])  # spin the pool up at this width
        dt = float("inf")
        for _ in range(3):
            t0 = time.perf_counter()
            fn(src, dst)
            dt = min(dt, time.perf_counter() - t0)
        if dt < best_t:
            best, best_t = n, dt
    orc.lib().orc_set_num_threads(best)
    return best, ncpu


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(device), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if sm:
            out = dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def ncu_traffic(kernel_family, workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    `ncu --set full` capture (profiles/traffic.json, written by profiles/extract_traffic.py)."""
    p = os.path.join(REPO, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        t = json.load(f)
    return t.get(workload, {}).get(kernel_family)


def traffic_fields(kernel_family, workload):
    """-> (`roofline.traffic`: bytes per launch or None, the capture's details)."""
    d = ncu_traffic(kernel_family, workload)
    if not d:
        return None, None
    return d.get("dram_bytes_per_launch"), d


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------------------------------
# the CPU arm (oracle port; kNN through the reference's own nanoflann when oracle/_ref is built)
# ---------------------------------------------------------------------------------------------------------------------
def oracle_setup():
    unbind_cpus()
    from oracle import oracle as orc
    orc.lib()
    used_ref = orc.use_ref_nanoflann(True) == 0
    return orc, used_ref


_LAST_THREADS = [None]


def run_cpu(fn, pairs, max_pairs, budget_s, what, orc, used_ref, calibrate=True):
    """Time fn(src, dst) on a bounded sample; returns (cpu_baseline dict, list of results).  calibrate=False reuses the thread
    count of the previous calibration (the raw 100k Quatro pair takes tens of seconds per call on the CPU)."""
    if calibrate or _LAST_THREADS[0] is None:
        threads, ncpu = calibrate_threads(orc, fn, pairs[0])
        _LAST_THREADS[0] = threads
    else:
        threads = _LAST_THREADS[0]
        ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        orc.lib().orc_set_num_threads(threads)
    times, outs = [], []
    t_start = time.perf_counter()
    for i in range(min(max_pairs, len(pairs))):
        t0 = time.perf_counter()
        outs.append(fn(pairs[i][0], pairs[i][1]))
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s:
            break
    per_pair = float(np.mean(times))
    return dict(value=1.0 / per_pair, unit=UNIT, cores=threads, logical_cpus=ncpu, kind="port",
                ms_per_pair=1e3 * per_pair, best_ms_per_pair=1e3 * float(np.min(times)),
                sample="%d pairs of %d x %d points, serial over pairs, OpenMP over points; restated %s (oracle/) with kNN = %s"
                       % (len(times), len(pairs[0][0]), len(pairs[0][1]), what,
                          "reference nanoflann (oracle/_ref)" if used_ref else "oracle kd-tree (oracle/_ref missing)"),
                cpu_model=cpu_info()[0]), outs


def main_reference(args):
    """The reference's CPU path on the SAME workload (config identical to the b200 arm, same seeds): every step is a
    bounded sample of the step's 256 pairs -- its first REF_PAIRS pairs, rotating through the rank-0 seeds."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    REF_PAIRS = 2
    n_distinct = min(JOB_PAIRS * DISTINCT_JOBS, REF_PAIRS * max(1, min(args.steps, 8)))
    pairs = gen_pairs(primary_seeds(0)[:n_distinct], args.points)
    orc, used_ref = oracle_setup()
    threads, ncpu = calibrate_threads(orc, orc.gicp_align, pairs[0])
    for w in range(max(args.warmup, 1)):
        orc.gicp_align(pairs[w % len(pairs)][0], pairs[w % len(pairs)][1])
    t0 = time.perf_counter()
    k = 0
    for _ in range(args.steps):
        for _ in range(REF_PAIRS):
            src, dst, _t = pairs[k % len(pairs)]
            orc.gicp_align(src, dst)
            k += 1
    dt = time.perf_counter() - t0
    val = REF_PAIRS * args.steps / dt
    sample = ("each step = the first %d pairs of the step's %d (seeds 1000..%d in rotation), run serially with all host threads "
              "per pair; CPU port of LoopClosure::icpAlignment with kNN = %s"
              % (REF_PAIRS, JOB_PAIRS * JOBS_PER_STEP, 1000 + len(pairs) - 1, "reference nanoflann (oracle/_ref)" if used_ref else "oracle kd-tree"))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 points+kNN / f64 covariance+solver", "data": "synthetic",
        "config": primary_config(args),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "logical_cpus": ncpu, "kind": "port", "sample": sample,
                         "cpu_model": cpu_info()[0]},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------------------------------------------------
# the b200 arm
# ---------------------------------------------------------------------------------------------------------------------
class Runner:
    """Timed regions over the C ABI's batch driver: CUDA events around, barrier + synchronize on both sides, max over ranks."""

    def __init__(self, batch, ctx, dist, stream, depth):
        self.batch, self.ctx, self.dist, self.stream, self.depth = batch, ctx, dist, stream, depth

    def run(self, n_jobs, submit, jobs_per_step=None, gather=False):
        """Submit n_jobs (at most 2*depth in flight), wait in order; after every jobs_per_step jobs all-gather that
        step's result records over the context's communicator.  Returns (ms, launches, results per job, job latencies)."""
        import torch
        from b200reg import native
        rebind_cpus()
        dist = self.dist
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = self.batch.launch_count + self.ctx.launch_count
        e0.record(self.stream)
        self.stream.synchronize()
        window = 2 * self.depth
        inflight, results, lats, step_buf, gathered = [], [], [], [], None
        nxt = 0
        while nxt < n_jobs or inflight:
            while nxt < n_jobs and len(inflight) < window:
                inflight.append(submit(nxt))
                nxt += 1
            res, lat = self.batch.wait(inflight.pop(0), want_latency=True)
            results.append(res)
            lats.append(lat)
            if gather and jobs_per_step:
                step_buf.append(res)
                if len(step_buf) == jobs_per_step:  # the ONE collective of the path: this step's result records
                    n = sum(len(r) for r in step_buf)
                    local = (native.Result * n)()
                    k = 0
                    for r in step_buf:
                        ctypes.memmove(ctypes.byref(local, k * ctypes.sizeof(native.Result)), r, ctypes.sizeof(r))
                        k += len(r)
                    gathered = self.ctx.allgather_results(local)
                    step_buf = []
        torch.cuda.synchronize()
        e1.record(self.stream)
        self.stream.synchronize()
        if dist is not None:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, self.batch.launch_count + self.ctx.launch_count - l0, results, lats, gathered


def check_accuracy(results, pairs, what):
    """The batch must land on its ground truth.  Individual synthetic pairs may legitimately defeat GICP itself (the CPU
    oracle diverges identically on them): they are counted and reported, never replaced; a batch that mostly fails
    means broken kernels and aborts the run."""
    from b200reg import synth
    worst = [0.0, 0.0]
    off = []
    for i, (r, p) in enumerate(zip(results, pairs)):
        rot, tr = synth.se3_error(np.array(r.T).reshape(4, 4), p[2])
        if not r.converged or rot > 1e-2 or tr > 0.1:
            off.append(i)
        else:
            worst = [max(worst[0], rot), max(worst[1], tr)]
    if len(off) > max(1, len(pairs) // 4):
        raise SystemExit("bench.py: %d of %d %s registrations missed the ground truth -- refusing to report a number" % (len(off), len(pairs), what))
    return dict(worst_rot_rad_vs_gt=worst[0], worst_trans_m_vs_gt=worst[1], pairs_off_ground_truth=off,
                mean_linearize_passes=float(np.mean([r.n_linearize for r in results])),
                max_linearize_passes=int(max(r.n_linearize for r in results)))


def parity_vs_oracle(gpu_results, cpu_results, what, gpu_T=lambda r: np.array(r.T).reshape(4, 4)):
    """GPU transforms against the CPU oracle's on the same pairs; aborts on a miss (the bar of BASELINE.json)."""
    from b200reg import synth
    worst = [0.0, 0.0]
    for i, (g, o) in enumerate(zip(gpu_results, cpu_results)):
        rot, tr = synth.se3_error(gpu_T(g), o["T"])
        worst = [max(worst[0], rot), max(worst[1], tr)]
        og = o.get("gicp", o)
        if rot > ROT_TOL or tr > TRANS_TOL or bool(g.converged) != bool(o["converged"]) or g.n_linearize != og["n_linearize"]:
            raise SystemExit("bench.py: %s parity miss on sampled pair %d: rot %.3e rad, trans %.3e m, converged %s/%s, linearize %d/%d"
                             % (what, i, rot, tr, bool(g.converged), o["converged"], g.n_linearize, og["n_linearize"]))
    return dict(pairs=len(cpu_results), worst_rot=worst[0], worst_trans=worst[1], counters_equal=True,
                tolerance="%g rad / %g m" % (ROT_TOL, TRANS_TOL))


DUMP_FIELDS = ("T", "Tf", "pose_between", "final_hessian", "fitness", "converged", "valid", "iterations", "n_linearize", "n_error",
               "lm_failed", "status")


def dump_outputs(directory, jobs):
    """One .npy per field of b200reg_result over every pair of `jobs` (lists of result records, in submission order): what
    the caller of b200reg_batch_wait receives.  Integer and flag fields are stored as float64."""
    recs = [r.as_dict() for job in jobs for r in job]
    os.makedirs(directory, exist_ok=True)
    for name in DUMP_FIELDS:
        a = np.array([d[name] for d in recs])
        np.save(os.path.join(directory, name + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


def percentiles(x):
    x = np.asarray(x, np.float64)
    return dict(p50=float(np.percentile(x, 50)), p99=float(np.percentile(x, 99)), max=float(x.max()), n=int(len(x)))


def family_table(prof, prof_steps):
    tot_ms = sum(v["ms"] for v in prof.values())
    return {k: dict(ms_per_step=v["ms"] / prof_steps, launches_per_step=v["launches"] / prof_steps,
                    algo_gb_per_step=v["algo_bytes"] / prof_steps / 1e9,
                    achieved_gbs=(v["algo_bytes"] / (v["ms"] * 1e-3) / 1e9) if v["ms"] > 0 else 0.0,
                    share=v["ms"] / tot_ms if tot_ms > 0 else 0.0) for k, v in prof.items() if v["ms"] > 0}


def profile_families(ctx, fn, reps):
    """Per-kernel-family CUDA-event timing on the launching stream (one context, so the families do not overlap)."""
    ctx.set_profiling(True)
    ctx.reset_profile()
    for i in range(reps):
        fn(i)
    prof = ctx.get_profile()
    ctx.set_profiling(False)
    return prof


def main():
    args = parse()
    if args.impl == "reference":
        return main_reference(args)

    import torch
    import b200reg
    from b200reg import native, synth

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the b200 arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    affinity = bind_near_gpu(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        saved = os.dup(1)
        os.dup2(2, 1)  # anything NCCL still prints while the communicator comes up goes to stderr
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            warm = torch.zeros(8, device="cuda")
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    sec = set() if args.secondary == "none" else set(("voxel,raw,sequence,batch512" if args.secondary == "all" else args.secondary).split(","))

    ctx = b200reg.Context(local_rank)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    if world > 1:  # the data-path collective lives behind the C ABI; the 128-byte id rides on the process group that is up
        box = [b200reg.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        ctx.comm_init(box[0], rank, world)
    batch = b200reg.Batch(local_rank, depth=args.depth)
    runner = Runner(batch, ctx, dist, stream, args.depth)
    prm = b200reg.default_params()
    qprm = native.default_quatro_params()
    qprm.use_optimized_matching = 1 if args.matching == "optimized" else 0
    res_bytes = ctypes.sizeof(native.Result)

    # ---- headline: configs[1] -----------------------------------------------------------------------------------------
    pairs = gen_pairs(primary_seeds(), args.points)
    arena = Arena(pairs, JOB_PAIRS)

    # the from-host arm runs on its own batch driver with more contexts (--depth-e2e): more uploads in flight
    batch_h = batch if args.depth_e2e == args.depth else b200reg.Batch(local_rank, depth=args.depth_e2e)
    runner_h = runner if batch_h is batch else Runner(batch_h, ctx, dist, stream, args.depth_e2e)

    def submit_icp(on_device):
        b = batch if on_device else batch_h
        return lambda j: b.submit_icp(*arena.job(j + rank, on_device), prm)

    sampler = ClockSampler(local_rank) if rank == 0 else None  # samples from the warm-up on: same load as the timed region
    # every context sees every sub-batch, both arms
    # (the warm-up includes the per-step gather: NCCL sets its channels up lazily on the first collective of a communicator)
    # Each arm: W (>= 3) full warm-up steps plus a fixed spin-up of SPIN_STEPS steps right before ITS timed region -- the
    # first process on a fresh box measured 30 % low for about a second (page-ins, memory pools, host threads waking up).
    SPIN_STEPS = 12
    n_warm = (max(args.warmup, 3) + SPIN_STEPS) * JOBS_PER_STEP
    n_jobs = args.steps * JOBS_PER_STEP
    runner.run(n_warm, submit_icp(True), JOBS_PER_STEP, gather=world > 1)
    ms_dev, launches, res_dev, lat_dev, _ = runner.run(n_jobs, submit_icp(True), JOBS_PER_STEP, gather=world > 1)
    runner_h.run(n_warm, submit_icp(False), JOBS_PER_STEP, gather=world > 1)
    ms_e2e, _, res_e2e, lat_e2e, _ = runner_h.run(n_jobs, submit_icp(False), JOBS_PER_STEP, gather=world > 1)
    if batch_h is not batch:
        batch_h.close()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:  # the last timed step of the device-resident arm: 16 jobs x 16 pairs
        dump_outputs(args.dump_outputs, res_dev[-JOBS_PER_STEP:])

    # one result per distinct pair (jobs 0..3 of the device arm), bit-identical across repeats and arms
    first = {(j + rank) % DISTINCT_JOBS: j for j in reversed(range(DISTINCT_JOBS))}  # sub-batch -> first job that ran it
    flat = [r for b in range(DISTINCT_JOBS) for r in res_dev[first[b]]]
    res_dev = res_dev[-rank % DISTINCT_JOBS:] if rank % DISTINCT_JOBS else res_dev  # re-align job j with sub-batch j % 4
    res_e2e = res_e2e[-rank % DISTINCT_JOBS:] if rank % DISTINCT_JOBS else res_e2e
    for j in range(DISTINCT_JOBS, min(len(res_dev), len(res_e2e))):
        if bytes(res_dev[j]) != bytes(res_dev[j % DISTINCT_JOBS]) or bytes(res_e2e[j]) != bytes(res_dev[j % DISTINCT_JOBS]):
            raise SystemExit("bench.py: repeated jobs over the same pairs returned different bytes (job %d)" % j)
    accuracy = check_accuracy(flat, pairs, "icpAlignment")
    accuracy["not_converged_seeds"] = [primary_seeds()[i] for i in accuracy.pop("pairs_off_ground_truth")]

    # per-kernel-family timing (one context, one 16-pair job at a time, rotating over the distinct sub-batches)
    prof_steps = 8
    prof = profile_families(ctx, lambda i: ctx.icp_alignment_ptrs(*arena.job(i, True), prm), prof_steps)

    out = None
    if rank == 0:
        total_pairs = world * JOB_PAIRS * n_jobs
        peak, peak_src = peaks()
        fam = max((k for k in prof if k != "misc"), key=lambda k: prof[k]["ms"])
        f = prof[fam]
        achieved = f["algo_bytes"] / (f["ms"] * 1e-3) / 1e9 if f["ms"] > 0 else 0.0
        cfg = primary_config(args)  # identical to the reference arm's
        parallelism = ("pairs sharded over %d ranks (256 per rank and step, the same 64-pair pool on every rank so that the per-GPU "
                       "work is fixed), no data-path collective but ONE ncclAllGather of the step's result records per step through "
                       "b200reg_allgather_results" % world) if world > 1 else "single GPU"
        out = {
            "metric": METRIC, "value": total_pairs / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 points+kNN / f64 covariance+solver", "data": "synthetic",
            "config": cfg, "parallelism": parallelism,
            "driver": "b200reg_batch (C ABI, csrc/batch.cu): %d engine contexts on C++ host threads, %d-pair jobs, at most %d jobs in flight "
                      "(from-host arm: %d contexts, %d jobs in flight)" % (args.depth, JOB_PAIRS, 2 * args.depth, args.depth_e2e, 2 * args.depth_e2e),
            "timed_region_s": ms_dev * 1e-3, "host_affinity": affinity,
            "lm_as_cuda_graph": not os.environ.get("B200REG_LM_NO_GRAPH"), "retried_after_failure": bool(os.environ.get("B200REG_BENCH_RETRIED")), "spin_up_steps_before_each_timed_region": SPIN_STEPS,
            "e2e": {"value": total_pairs / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": sum(arena.h2d_bytes(j) for j in range(JOBS_PER_STEP)),
                    "d2h_bytes_per_step": JOB_PAIRS * JOBS_PER_STEP * res_bytes, "timed_region_s": ms_e2e * 1e-3},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": fam, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic_fields(fam, "gicp")[0], "traffic_unit": "bytes per launch",
                         "traffic_capture": traffic_fields(fam, "gicp")[1], "algorithmic_bytes_per_launch": f["algo_bytes"] / max(1, f["launches"]),
                         "peak_source": peak_src,
                         "note": "dominant KERNEL of the step (largest total CUDA-event time among the kernels / single-kernel families): "
                                 "algorithmic bytes per SURVEY.md §8(d) / its CUDA-event time on the launching stream, %d profiled 16-pair jobs "
                                 "on one context after the timed region; while profiling, the LM loop's three kernels are launched one by one "
                                 "instead of as one graph so that each gets its own events" % prof_steps},
            "kernels": family_table(prof, prof_steps),
            "clocks": clocks,
            "accuracy": accuracy,
            "job_latency_ms_under_load": {"device_resident": percentiles(lat_dev), "from_host": percentiles(lat_e2e),
                                          "note": "submit -> completion of one 16-pair job with up to %d (device_resident) / %d (from_host) "
                                                  "jobs in flight" % (2 * args.depth, 2 * args.depth_e2e)},
        }

    # ---- single-pair latency through ONE C-ABI call on an idle GPU (the reference's "ms per ICP" view) ---------------------
    if rank == 0:
        lat1 = []
        for i in range(32):
            k = (2 * i) % len(arena.hs)
            hs, hd = arena.hs[k], arena.hd[k]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ctx.icp_alignment_ptrs([hs.data_ptr()], [hs.shape[0]], [hd.data_ptr()], [hd.shape[0]], arena.stride, 0, prm)
            lat1.append(1e3 * (time.perf_counter() - t0))
        out["latency"] = {"single_pair_icp_alignment_ms": percentiles(lat1[2:]),
                          "note": "one 100k x 100k pair per b200reg_icp_alignment call from pinned host buffers, idle GPU, wall clock around the "
                                  "call (upload, 2 index builds, 2 covariance passes, LM, fitness, result read-back): what NanoGICP::align's "
                                  "caller times in fast_lio_sam_qn.cpp:212-243"}

    # ---- CPU oracle on a bounded sample of the same pairs + parity of the GPU transforms against it ------------------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        orc, used_ref = oracle_setup()
        out["cpu_baseline"], cpu_res = run_cpu(orc.gicp_align, pairs, args.cpu_sample_pairs, 20.0, "Nano-GICP", orc, used_ref)
        par = parity_vs_oracle(flat[:len(cpu_res)], cpu_res, "icpAlignment")
        # correspondences of the first linearize of pair 0: bit-exact indices and fp32 distances at 100k x 100k
        cs, ct = ctx.create_clouds([pairs[0][0], pairs[0][1]])
        ctx.covariances([cs, ct], 15)
        lin = ctx.linearize(cs, ct, np.eye(4))
        ol = orc.linearize(pairs[0][0], pairs[0][1], ctx.get_covariances(cs), ctx.get_covariances(ct), np.eye(4))
        par["corr_exact"] = bool(np.array_equal(lin["corr"], ol["corr"]) and np.array_equal(lin["sqd"], ol["sqd"]))
        cs.destroy(); ct.destroy()
        if not par["corr_exact"]:
            raise SystemExit("bench.py: first-linearize correspondences differ from the oracle's")
        out["parity"] = par

    # ---- secondary workloads -------------------------------------------------------------------------------------------
    # (a failure in one of them must not take the headline with it: it is recorded and the line is printed)
    secondary = {}
    try:
        run_secondaries(args, sec, secondary, world, rank, local_rank, runner, batch, ctx, dist, stream, qprm, prm, pairs)
    except BaseException as e:  # noqa: BLE001
        if isinstance(e, KeyboardInterrupt):
            raise
        import traceback
        traceback.print_exc()
        secondary["failed"] = "%s: %s" % (type(e).__name__, e)
        if rank == 0:
            out["secondary"] = secondary
            print(json.dumps(out))
            sys.stdout.flush()
        os._exit(0 if world == 1 else 1)  # the CUDA context may be unusable: no teardown
    if rank == 0:
        if secondary:
            out["secondary"] = secondary
        print(json.dumps(out))
    batch.close()
    if dist is not None:
        dist.barrier()
    if world > 1:
        ctx.comm_destroy()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


def run_secondaries(args, sec, secondary, world, rank, local_rank, runner, batch, ctx, dist, stream, qprm, prm, pairs):
    import b200reg
    if world == 1:
        if "voxel" in sec or "raw" in sec:
            own = args.depth_lc != args.depth
            batch_lc = b200reg.Batch(local_rank, depth=args.depth_lc) if own else batch
            runner_lc = Runner(batch_lc, ctx, dist, stream, args.depth_lc) if own else runner
        if "voxel" in sec:
            secondary["loop_closure_voxelised"] = bench_loop_closure(args, runner_lc, batch_lc, ctx, qprm, prm, voxel=0.3, n_pairs=64,
                                                                     per_job=16, jobs=192, cpu_pairs=3)
        if "raw" in sec:
            secondary["loop_closure_raw_100k"] = bench_loop_closure(args, runner_lc, batch_lc, ctx, qprm, prm, voxel=None, n_pairs=8, per_job=4,
                                                                    jobs=16, cpu_pairs=1)
        if ("voxel" in sec or "raw" in sec) and own:
            batch_lc.close()
        if "sequence" in sec:
            secondary["sequence_kitti05_shaped"] = bench_sequence(args, ctx, stream)
    else:
        if "batch512" in sec:
            secondary["batch_512_pairs_sharded"] = bench_batch512(args, runner, batch, ctx, dist, prm, rank, world)
            secondary["rank_distinct_pools"] = bench_rank_distinct(args, runner, batch, prm, rank, world, pairs)


def bench_loop_closure(args, runner, batch, ctx, qprm, prm, voxel, n_pairs, per_job, jobs, cpu_pairs):
    """configs[2]: LoopClosure::coarseToFineAlignment (FPFH -> matching -> QUATRO solve -> transform -> GICP refine),
    SURVEY §8(d) seeds 2000..., on scans voxelised at 0.3 m like setSrcAndDstCloud (loop_closure.cpp:107) or RAW."""
    from b200reg import native
    pairs = gen_pairs([2000 + i for i in range(n_pairs)], args.points, mode="quatro", voxel=voxel)
    arena = Arena(pairs, per_job)

    def submit(on_device):
        return lambda j: batch.submit_loop_closure(*arena.job(j, on_device), qprm, prm)
    njobs_distinct = len(arena.jobs)
    runner.run(max(njobs_distinct, 2 * runner.depth), submit(True))
    runner.run(max(njobs_distinct, 2 * runner.depth), submit(False))
    ms_dev, launches, res, lat, _ = runner.run(jobs, submit(True))
    ms_e2e, _, _, lat_h, _ = runner.run(jobs, submit(False))
    flat = [r for j in range(njobs_distinct) for r in res[j]]
    acc = check_accuracy(flat, pairs, "coarse-to-fine")
    acc["not_converged_seeds"] = [2000 + i for i in acc.pop("pairs_off_ground_truth")]
    prof = profile_families(ctx, lambda i: ctx.loop_closure_ptrs(*arena.job(i, True), qprm, prm), njobs_distinct)
    sizes = [len(p[0]) for p in pairs] + [len(p[1]) for p in pairs]
    out = {"metric": "full_loop_closure_registrations_per_sec", "unit": UNIT,
           "workload": "configs[2]: Quatro+Nano-GICP full loop closure (LoopClosure::coarseToFineAlignment, %sMatching) on %s"
                       % (args.matching, ("%dk-pt scans voxelised at %.1f m" % (args.points // 1000, voxel)) if voxel else
                          ("RAW %dk x %dk-pt scans (no voxel grid)" % (args.points // 1000, args.points // 1000))),
           "points_per_cloud": {"min": int(min(sizes)), "median": int(np.median(sizes)), "max": int(max(sizes))},
           "distinct_pairs": n_pairs, "pairs_per_job": per_job, "jobs_timed": jobs, "seeds": "2000 + i", "driver_contexts": runner.depth,
           "value": per_job * jobs / (ms_dev * 1e-3), "timed_region_s": ms_dev * 1e-3,
           "e2e": {"value": per_job * jobs / (ms_e2e * 1e-3), "unit": UNIT,
                   "h2d_bytes_per_job": arena.h2d_bytes(0), "d2h_bytes_per_job": per_job * (ctypes.sizeof(native.Result) + ctypes.sizeof(native.QuatroInfo))},
           "gpu_launches": launches, "kernels": family_table(prof, njobs_distinct), "accuracy": acc,
           "job_latency_ms_under_load": percentiles(lat)}
    if not args.no_cpu_baseline:
        orc, used_ref = oracle_setup()
        qp = orc.QuatroParams.default()
        qp.use_optimized_matching = 1 if args.matching == "optimized" else 0
        out["cpu_baseline"], cpu_res = run_cpu(lambda s, d: orc.coarse_to_fine(s, d, qparams=qp), pairs, cpu_pairs, 40.0,
                                               "Quatro (FPFH + brute-force 33-D matching + QUATRO solve) + Nano-GICP", orc, used_ref,
                                               calibrate=voxel is not None)
        # parity at the bar: the fine stage on the SAME coarse transform (the two coarse stages differ by fp32 summation order
        # of the descriptors and are only required to agree to the refinement's basin, tests/test_gpu_quatro.py)
        single, qi = ctx.loop_closure([p[0] for p in pairs[:len(cpu_res)]], [p[1] for p in pairs[:len(cpu_res)]], qparams=qprm, gparams=prm)
        same = [orc.coarse_to_fine(p[0], p[1], qparams=qp, quatro_T=q["T"]) for p, q in zip(pairs, qi)]

        class _R:  # adapter: dict -> attribute access
            def __init__(self, d):
                self.T, self.converged, self.n_linearize = d["T"].reshape(-1), d["converged"], d["n_linearize"]
        out["parity"] = parity_vs_oracle([_R(r) for r in single], same, "coarse-to-fine (fine stage on the same coarse transform)")
        from b200reg import synth
        pipe = [synth.se3_error(r["T"], o["T"]) for r, o in zip(single, cpu_res)]
        out["parity"]["complete_pipelines_worst_rot"] = float(max(p[0] for p in pipe))
        out["parity"]["complete_pipelines_worst_trans"] = float(max(p[1] for p in pipe))
    return out


def bench_sequence(args, ctx, stream):
    """configs[4]: every keyframe of a synthetic KITTI-05-shaped sequence that has a loop candidate goes through
    fetchClosestKeyframeIdx + setSrcAndDstCloud + coarse-to-fine registration, all from device-resident keyframes
    (loopTimerFunc, fast_lio_sam_qn.cpp:203-252)."""
    import torch
    import b200reg
    from b200reg import synth
    B = 16
    pts = 30000  # ~120k returns / 4 (kitti.launch:7)
    seq = synth.make_sequence(5, args.keyframes, pts_per_keyframe=pts, threads=max(1, (os.cpu_count() or 8) // 8))
    kf = ctx.keyframes()
    kf.reserve(sum(len(c) for c in seq["clouds"]))
    for c, T, t in zip(seq["clouds"], seq["poses"], seq["stamps"]):
        kf.add(c, T, t)
    ctx.synchronize()
    cfg = b200reg.default_loop_config()
    allq = np.arange(args.keyframes, dtype=np.int32)
    closest_all = kf.fetch_closest(allq, cfg.loop_detection_radius, cfg.loop_detection_timediff_threshold)
    cand = allq[closest_all >= 0]
    if len(cand) < B:
        kf.destroy()
        return {"unavailable": "sequence too short for loop candidates (%d)" % len(cand)}
    batches = [cand[i:i + B] for i in range(0, len(cand) - B + 1, B)]
    pinned = [torch.from_numpy(seq["clouds"][q]).pin_memory() for q in cand[:B]]

    def step(i, ingest):
        q = batches[i % len(batches)]
        if ingest:  # e2e: the step's query keyframes arrive from the host first (odomPcdCallback -> keyframe store)
            for j, qq in enumerate(q):
                kf.add(pinned[j % len(pinned)].numpy(), seq["poses"][qq], seq["stamps"][qq])
        cl = kf.fetch_closest(q, cfg.loop_detection_radius, cfg.loop_detection_timediff_threshold)
        return kf.perform_loop_closure(q, cl, cfg, raw=True)

    def timed(ingest, steps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count
        nvalid = 0
        with torch.cuda.stream(stream):
            e0.record(stream)
            for i in range(steps):
                out = step(i, ingest)
                nvalid += sum(1 for r in out[0] if r.valid)
            e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), ctx.launch_count - l0, nvalid

    for i in range(3):
        step(i, False)
    steps = len(batches)  # every candidate of the sequence exactly once
    ms_dev, launches, nvalid = timed(False, steps)
    # the ingest path: the node reserves the device room of its map once (b200reg_keyframes_reserve), as a long-running node
    # does; then spin-up steps as for the headline (a fresh box answers slowly for its first second)
    e2e_steps = min(steps, 48)
    kf.reserve(B * (e2e_steps + 24) * pts)
    for i in range(20):
        step(i, True)
    ms_e2e, _, _ = timed(True, e2e_steps)
    prof = profile_families(ctx, lambda i: step(i, False), min(4, steps))
    res = {"metric": "loop_closure_attempts_per_sec_kitti05_shaped_sequence", "unit": UNIT,
           "workload": "configs[4]: loopTimerFunc over a synthetic KITTI-05-shaped sequence of %d keyframes x %dk points kept on the device: "
                       "fetchClosestKeyframeIdx + setSrcAndDstCloud (transform, voxel 0.3 m) + Quatro + Nano-GICP for EVERY keyframe that has a "
                       "loop candidate, %d per call" % (args.keyframes, pts // 1000, B),
           "keyframes": args.keyframes, "candidates": int(len(cand)), "attempts_timed": B * steps, "valid_loops": int(nvalid),
           "value": B * steps / (ms_dev * 1e-3), "timed_region_s": ms_dev * 1e-3, "ms_per_attempt": ms_dev / (B * steps),
           "e2e": {"value": B * e2e_steps / (ms_e2e * 1e-3), "unit": UNIT, "calls_timed": e2e_steps, "h2d_bytes_per_call": B * pts * 16,
                   "d2h_bytes_per_call": B * ctypes.sizeof(b200reg.Result),
                   "note": "the 16 query keyframes of every call are ingested from pinned host memory first"},
           "gpu_launches": launches, "kernels": family_table(prof, min(4, steps))}
    if not args.no_cpu_baseline:
        orc, used_ref = oracle_setup()
        q0 = batches[0]
        c0 = kf.fetch_closest(q0)
        pair0 = orc.set_src_and_dst_cloud(seq["clouds"], seq["poses"], int(q0[0]), int(c0[0]), n_keyframes=int(q0[0]) + 1)
        threads, ncpu = calibrate_threads(orc, lambda a, b: orc.coarse_to_fine(a, b), pair0)
        t0 = time.perf_counter()
        nrun = 0
        for qq, cc in zip(q0[:6], c0[:6]):
            pos = seq["poses"][:int(qq) + 1, :3, 3]
            orc.fetch_closest(pos, seq["stamps"], int(qq))
            s_, d_ = orc.set_src_and_dst_cloud(seq["clouds"], seq["poses"], int(qq), int(cc), n_keyframes=int(qq) + 1)
            orc.coarse_to_fine(s_, d_)
            nrun += 1
        dt = time.perf_counter() - t0
        res["cpu_baseline"] = {"value": nrun / dt, "unit": UNIT, "cores": threads, "logical_cpus": ncpu, "kind": "port",
                               "sample": "%d loop attempts (candidate search + assembly + Quatro + GICP), CPU oracle" % nrun,
                               "cpu_model": cpu_info()[0]}
    kf.destroy()
    return res


def bench_rank_distinct(args, runner, batch, prm, rank, world, pool0):
    """The headline's region with a DIFFERENT 64-pair pool on every rank (seeds 1000 + 64*rank + i): the pools differ in
    cost, every step ends with the all-gather, so the heaviest pool sets the pace -- data skew, reported beside the
    fixed-work headline rather than inside it."""
    import torch
    pairs = pool0 if rank == 0 else gen_pairs(rank_distinct_seeds(rank), args.points)
    arena = Arena(pairs, JOB_PAIRS)
    steps = 6

    def submit(j):
        return batch.submit_icp(*arena.job(j, True), prm)
    runner.run(2 * DISTINCT_JOBS, submit, 2 * DISTINCT_JOBS, gather=True)
    ms, _, res, _, _ = runner.run(steps * JOBS_PER_STEP, submit, JOBS_PER_STEP, gather=True)
    mine = torch.tensor([float(np.mean([r.n_linearize for j in range(DISTINCT_JOBS) for r in res[j]])),
                         float(max(r.n_linearize for j in range(DISTINCT_JOBS) for r in res[j]))], dtype=torch.float64, device="cuda")
    allr = [torch.zeros_like(mine) for _ in range(world)]
    runner.dist.all_gather(allr, mine)
    if rank != 0:
        return None
    return {"metric": METRIC, "unit": UNIT, "value": world * JOB_PAIRS * steps * JOBS_PER_STEP / (ms * 1e-3), "steps": steps,
            "ms_per_step": ms / steps, "seeds": "1000 + 64*rank + i, i < 64", "inputs": "resident in HBM",
            "linearize_passes_per_rank": [{"mean": float(t[0]), "max": int(t[1])} for t in allr],
            "note": "same region as the headline with rank-distinct pools: the slowest pool bounds every step"}


def bench_batch512(args, runner, batch, ctx, dist, prm, rank, world):
    """configs[3]: ONE batch of 512 keyframe-pair candidates (SURVEY §8(d) seeds 3000...3511) sharded over the ranks in
    contiguous blocks (b200reg/sharding.py), registered in 16-pair jobs, then ONE ncclAllGather of the 512 result
    records (b200reg_allgather_results).  Strong scaling: the batch is fixed, the shard shrinks with N."""
    from b200reg import native
    from b200reg.sharding import shard_pairs
    mine = shard_pairs(512, world, rank)
    pairs = gen_pairs([3000 + i for i in mine], args.points)
    arena = Arena(pairs, JOB_PAIRS)
    njobs = len(arena.jobs)
    reps = 3

    def submit(j):
        return batch.submit_icp(*arena.job(j, True), prm)
    runner.run(njobs, submit, njobs, gather=True)  # warm-up
    ms = []
    for _ in range(reps):
        m, launches, res, _, gathered = runner.run(njobs, submit, njobs, gather=True)
        ms.append(m)
    if rank != 0:
        return None
    recs = list(gathered)
    T_ok = sum(1 for r in recs if r.converged)
    return {"metric": "batch_512_registrations_per_sec", "unit": UNIT,
            "workload": "configs[3]: batch of 512 keyframe-pair loop candidates (%dk x %dk points, seeds 3000..3511) sharded over %d GPUs, "
                        "%d pairs per rank, one ncclAllGather of the 512 result records (%d bytes each) per batch"
                        % (args.points // 1000, args.points // 1000, world, len(mine), ctypes.sizeof(native.Result)),
            "scaling": "strong", "value": 512.0 / (min(ms) * 1e-3), "ms_per_batch": {"best": min(ms), "all": ms},
            "gathered_records": len(recs), "converged": T_ok, "inputs": "resident in HBM", "gpu_launches_rank0": launches}


if __name__ == "__main__":
    try:
        main()
    except BaseException as e:  # noqa: BLE001
        if isinstance(e, SystemExit) and e.code in (0, None):
            raise
        import traceback
        traceback.print_exc()
        sys.stderr.flush()
        sys.stdout.flush()
        # One retry in a fresh process (single-GPU runs only: under torchrun the ranks cannot restart on their own).  Deliberate
        # aborts (SystemExit: parity miss, wrong results) are never retried.
        if (not isinstance(e, SystemExit) and os.environ.get("WORLD_SIZE", "1") == "1" and not os.environ.get("B200REG_BENCH_RETRIED")
                and "--impl" not in " ".join(sys.argv[1:]).replace("--impl b200", "")):
            os.environ["B200REG_BENCH_RETRIED"] = "1"
            os.environ["B200REG_LM_NO_GRAPH"] = "1"  # the retry launches the LM kernels one by one (no conditional graph nodes)
            sys.stderr.write("bench.py: the run failed before its JSON line was printed -- retrying ONCE in a fresh process, "
                             "without the LM graph\n")
            sys.stderr.flush()
            os.execv(sys.executable, [sys.executable] + sys.argv)
        # a rank that fails must not linger in destructors that wait for its peers (communicator teardown): exit hard, the
        # launcher then stops the other ranks
        os._exit(1 if not isinstance(e, SystemExit) else (e.code if isinstance(e.code, int) else 1))
