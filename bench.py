#!/usr/bin/env python3
"""bench.py -- registrations/sec of the VGICP hot path on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c2_direct1|c3|c4|c4_direct1|c5]
                    [--dump-outputs DIR]

Workload (N=1 default, BASELINE configs[1]): the reference's benchmark pair (tests/golden/pair_0p1.npz = data/251370668.pcd
vs 251371071.pcd after align.cpp's filter + ApproximateVoxelGrid(0.1): 17047 / 17334 points), FastVGICPCuda, DIRECT27,
voxel_res 1.0, k=20, PLANE, LM defaults, identity initial guess.

One registration follows the reference's "100times" protocol (src/align.cpp:72-81): clearTarget, clearSource,
setInputTarget (upload, kNN, covariances, voxel map), setInputSource (upload, kNN, covariances), align.
One *step* = one registration on each of S concurrent streams of the GPU (--streams, default 8 at every N: one host thread and one
handle per stream; a 17k-pt registration is a chain of small latency-bound kernels, so one stream cannot fill 148 SMs; the rate
saturates at 8 streams).  Host threads are pinned to the cores of the GPU's NUMA node, an own slice per rank.

  value  : registrations/s with the clouds already resident in HBM when the timed region starts (device pointers
           through the C ABI); device time from a common start event to the last stream's end event; every registration
           takes the next pair of a pool of distinct pairs that is larger than the L2.
  e2e    : the same through the reference-facing class FastVGICPCuda with HOST (pinned) buffers: H2D of both clouds and D2H
           of the aligned cloud + pose inside the timed region.
  single_stream: the sequential protocol on one stream (latency), L2 flushed between registrations.
  roofline: dominant kernel group of the step, algorithmic bytes (SURVEY.md 8d) / CUDA-event time, against MEASURED_PEAKS.json;
           traffic = ncu DRAM bytes (profiles/traffic.json, quoted only while it matches the CUDA sources being run).
  cpu_baseline: the reference's own CPU implementation of the path (OpenMP FastVGICP, restated in oracle/ because the
           reference cannot be compiled here) on 32 pinned host cores, median of >= 30 registrations; plus the FastGICP single-thread
           row of BASELINE config 1.
  published_configurations: the same pair as the reference's README rows run it (DIRECT1; DIRECT1 with RBF covariances).
  c4     : BASELINE config 4, the 1M-point pair: stage times and the evaluation kernel's HBM roofline (DIRECT27 and DIRECT1) on one
           GPU; with N > 1 the same registration with stage 1 and stage 3 sharded over the N ranks (in-kernel NVLink exchanges),
           speed-up against the unsharded registration measured in the same run, agreement and bit-identity across ranks.

--dump-outputs DIR (rank 0): what the timed registrations of the last step returned, one registration per stream, as DIR/<name>.npy
(float64 unless noted; the inputs are the same from run to run, so two builds can be compared output for output):
  pose, hessian       (S,4,4), (S,6,6): final transformation and Hessian of the resident arm (vgicp_register)
  counters            (S,5): nr_iterations, converged, n_linearize, n_compute_error, lm_failed of the same registrations
  e2e_pose            (S,4,4): final transformation of the e2e arm
  e2e_aligned         (S,n,3) float32: the aligned source clouds the e2e arm read back; above 16 MB a fixed seeded sample of n rows,
                      the same for every stream, whose indices are in e2e_aligned_rows (n,)

N>1 (torchrun): the 17k-pt path does not shard usefully (SURVEY 8e) -> replicas, S registration streams per GPU, no
data-path collective; value = N*S*K registrations / max-over-ranks time ("weak" scaling).  The c4 record is the sharded path.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# 8 handles x 2 streams alias onto the default 8 hardware work queues and wait on each other; 32 queues (read by the driver when the context is
# created) give +5..9 % registrations/s at 8 handles, +20 % at 16 (profiles/r02_connections_sweep.txt).  fast_gicp_b200.core sets the same default.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

_REAL_STDOUT = sys.stdout
METRIC = "registrations/sec (VGICP, ~17k-pt pairs)"
UNIT = "registrations/s"


# ------------------------------------------------------------------------------------------------------------ inputs
def load_workload(name):
    if name in ("c2", "c2_direct1"):
        d = np.load(os.path.join(ROOT, "tests", "golden", "pair_0p1.npz"))
        return dict(
            name="C2: FastVGICPCuda %s res=1.0 k=20 PLANE LM, 17k-pt fixture pair (17047/17334 pts)" % ("DIRECT27" if name == "c2" else "DIRECT1"),
            target=np.ascontiguousarray(d["target"], dtype=np.float32), source=np.ascontiguousarray(d["source"], dtype=np.float32),
            method="DIRECT27" if name == "c2" else "DIRECT1", res=1.0,
            data="fixture: reference data/251370668.pcd vs 251371071.pcd, align.cpp filter + ApproximateVoxelGrid(0.1)")
    from fast_gicp_b200.synthetic import kitti_like_pair

    if name == "c3":
        t, s, _ = kitti_like_pair(beams=64, az_steps=2083, seed=42, pose=(0.8, 0.05, 0.7), downsample=0.25)
        return dict(name="C3: synthetic HDL-64 pair (0.25 m downsample) DIRECT27 res=1.0", target=t, source=s, method="DIRECT27", res=1.0, data="synthetic")
    if name == "c5":
        t, s, _ = kitti_like_pair(beams=64, az_steps=2083, seed=1000, pose=(0.8, 0.05, 0.7), downsample=0.25)
        return dict(name="C5: NDTCuda D2D DIRECT7 res=1.0, synthetic HDL-64 pair (0.25 m downsample)", target=t, source=s, method="DIRECT7", res=1.0, data="synthetic",
                    problem="ndt_d2d")
    if name in ("c4", "c4_direct1"):
        t, s, _ = kitti_like_pair(beams=128, az_steps=8192, seed=44, pose=(0.5, 0.0, 1.0), downsample=0.0, max_points=1_000_000)
        method = "DIRECT27" if name == "c4" else "DIRECT1"  # DIRECT1: the bandwidth-bound configuration of the evaluation kernel (DESIGN.md 4)
        return dict(name="C4: synthetic 1M-pt pair %s res=0.5" % method, target=t, source=s, method=method, res=0.5, data="synthetic")
    raise SystemExit("unknown workload " + name)


# --------------------------------------------------------------------------------------------------- clocks sampling
class ClockSampler:
    FIELDS = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(prefix="clocks_", suffix=".csv")
        self.proc = None
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            p = [x.strip() for x in line.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for nme, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# -------------------------------------------------------------------------------------------------------- CPU arm
def numa_cpus(node):
    """One hardware thread per physical core of a NUMA node (sysfs), or None."""
    try:
        txt = open("/sys/devices/system/node/node%d/cpulist" % node).read().strip()
        cpus = []
        for part in txt.split(","):
            lo, _, hi = part.partition("-")
            cpus.extend(range(int(lo), int(hi or lo) + 1))
        seen, out = set(), []
        for c in cpus:
            try:
                sib = open("/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list" % c).read().strip()
            except OSError:
                sib = str(c)
            if sib not in seen:
                seen.add(sib)
                out.append(c)
        return out or None
    except (OSError, ValueError):
        return None


def cpu_thread_set():
    """The CPU arm's threads: the physical cores of NUMA node 0 (capped at 32: OpenMP over ~17k points stops scaling there), fixed
    and pinned, so that two runs on two boxes of the same class measure the same thing."""
    allowed = sorted(os.sched_getaffinity(0))
    cpus = [c for c in (numa_cpus(0) or allowed) if c in allowed] or allowed
    return cpus[:32]


def cpu_one_registration(w, offs, threads):
    import oracle as O

    tgt, src = w["target"], w["source"]
    if w.get("problem") == "ndt_d2d":  # the reference has no CPU NDT of its own: the float restatement of NDTCuda serves as the CPU arm
        return O.register_ndt(tgt, src, res=w["res"], mode=O.D2D, method=getattr(O, w["method"]))
    tc = O.covariances_f64(tgt, 20, O.REG_PLANE, threads)
    sc = O.covariances_f64(src, 20, O.REG_PLANE, threads)
    return O.align_f64(tgt, tc, src, sc, res=w["res"], offs=offs, threads=threads)


def run_reference_arm(args, w, rank, world):
    """--impl reference: the reference's CPU implementation of this path (OpenMP FastVGICP, restated in oracle/ because the
    reference cannot be compiled here: per registration calculate_covariances(target), calculate_covariances(source) (kd-tree
    kNN, k=20, PLANE), voxel map, LM align) on a fixed, pinned set of host cores; rank 0 only.  A step is a bounded sample of
    `regs_per_step` registrations (so that even a short --steps run times >= 30 of them); value = 1 / median registration time."""
    if rank != 0:
        return
    cpus = cpu_thread_set()
    # the OpenMP runtime reads these when the oracle library loads (first use below)
    os.environ.setdefault("OMP_PROC_BIND", "true")
    os.environ["OMP_PLACES"] = ",".join("{%d}" % c for c in cpus)
    os.environ["OMP_NUM_THREADS"] = str(len(cpus))
    os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
    try:
        os.sched_setaffinity(0, cpus)
    except OSError:
        pass
    import oracle as O

    offs = O.offsets(getattr(O, w["method"]))
    threads = len(cpus)
    per_step = max(1, -(-30 // max(args.steps, 1)))
    for _ in range(max(args.warmup, 3)):
        cpu_one_registration(w, offs, threads)
    times = []
    for _ in range(args.steps * per_step):
        t0 = time.perf_counter()
        cpu_one_registration(w, offs, threads)
        times.append(time.perf_counter() - t0)
    med = float(np.median(times))
    value = 1.0 / med
    # BASELINE config 1: FastGICP, single thread (fast_gicp_impl.hpp:117-301 restated), same pair; a reported row, not the arm's value
    config1 = None
    if w.get("problem") != "ndt_d2d" and len(w["target"]) < 100000:
        t1 = []
        for _ in range(3):
            t0 = time.perf_counter()
            tc = O.covariances_f64(w["target"], 20, O.REG_PLANE, 1)
            sc = O.covariances_f64(w["source"], 20, O.REG_PLANE, 1)
            O.align_gicp_f64(w["target"], tc, w["source"], sc, threads=1)
            t1.append(time.perf_counter() - t0)
        config1 = {"value": 1.0 / float(np.median(t1)), "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": "3 registrations (median), restated FastGICPSingleThread (k-d tree k=20 covariances + point-to-point GICP, LM), published 9.4 registrations/s on an i9-9900K (README.md:121-122)"}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": 1e3 * med * per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": w["data"],
        "config": {"workload": w["name"], "protocol": "align.cpp 100times (covariances recomputed every registration)", "step": "%d sequential registrations" % per_step,
                   "registrations_timed": len(times), "statistic": "1 / median registration time", "mean_ms": 1e3 * float(np.mean(times)), "min_ms": 1e3 * float(np.min(times)),
                   "host_cores": os.cpu_count(), "pinned_cpus": "%d-%d (%d threads, one per physical core of NUMA node 0)" % (cpus[0], cpus[-1], threads)},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d full registrations (median), restated OpenMP FastVGICP in double (reference not buildable here: no Eigen/PCL), %d pinned threads" % (len(times), threads),
                         "config1_fastgicp_single_thread": config1},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_REAL_STDOUT, flush=True)


# ------------------------------------------------------------------------------------------------ host placement
def gpu_numa_node(torch, local_rank):
    try:
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(local_rank), "pci_domain_id", 0)
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        return node if node >= 0 else None
    except Exception:  # noqa: BLE001
        return None


def pin_rank_threads(torch, local_rank, world):
    """Keep this rank's host threads (one per registration stream) on cores of its GPU's NUMA node, an own slice per rank: with 8
    ranks x 8 spinning threads on two sockets the scheduler otherwise migrates them across nodes (SCALE_r01: e2e efficiency 0.81)."""
    node = gpu_numa_node(torch, local_rank)
    if node is None:
        return None
    try:
        txt = open("/sys/devices/system/node/node%d/cpulist" % node).read().strip()
        cpus = []
        for part in txt.split(","):
            lo, _, hi = part.partition("-")
            cpus.extend(range(int(lo), int(hi or lo) + 1))
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        n_gpus = torch.cuda.device_count()
        same = [g for g in range(n_gpus) if gpu_numa_node(torch, g) == node] or [local_rank]
        if world > 1 and len(same) > 1 and local_rank in same:
            j, m = same.index(local_rank), len(same)
            phys = len(cpus) // 2 if len(cpus) >= 2 * m else len(cpus)  # cpulist = physical cores then their hyper-thread siblings
            per = max(phys // m, 1)
            mine = cpus[j * per:(j + 1) * per]
            if phys < len(cpus):
                mine = mine + cpus[phys + j * per:phys + (j + 1) * per]
            cpus = mine or cpus
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": "%d..%d (%d)" % (cpus[0], cpus[-1], len(cpus))}
    except Exception:  # noqa: BLE001
        return None


def source_hash():
    """Hash of the CUDA sources: profiles/traffic.json (ncu DRAM bytes per launch) is only quoted while it matches."""
    import hashlib

    h = hashlib.sha256()
    d = os.path.join(ROOT, "fast_gicp_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".hpp")):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


# --------------------------------------------------------------------------------------------- C4 (1M-point pair)
def c4_record(torch, dev, local_rank, rank, world, peak_gbs, note):
    """BASELINE config 4: synthetic 1M-pt pair, res 0.5.  One GPU: stage times and the evaluation kernel against the HBM roofline
    (DIRECT1 = the bandwidth-bound configuration, DIRECT27 = the issue-bound one).  Several GPUs: the same registration with the
    source sharded over the ranks -- stage 1 (k-NN queries + covariances, exchanged by peer stores) and stage 3 (evaluation, 28 sums
    exchanged inside the kernel over NVLink peer memory) -- against the unsharded one measured in the same run."""
    from fast_gicp_b200 import distributed as D
    from fast_gicp_b200.core import REG_PLANE, Core, pose_from_c
    from fast_gicp_b200.synthetic import kitti_like_pair

    tgt, src, _ = kitti_like_pair(beams=128, az_steps=8192, seed=44, pose=(0.5, 0.0, 1.0), downsample=0.0, max_points=1_000_000)
    n_t, n_s = len(tgt), len(src)
    d_t, d_s = torch.from_numpy(tgt).to(dev), torch.from_numpy(src).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def registration(c, timed=True):
        st = torch.cuda.ExternalStream(c.stream(), device=dev)
        flush.zero_()
        torch.cuda.synchronize()
        D.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        c.set_cloud_device("target", d_t.data_ptr(), n_t, 12)
        c.find_target_neighbors(20)
        c.calculate_target_covariances(REG_PLANE)
        c.create_target_voxelmap()
        c.set_cloud_device("source", d_s.data_ptr(), n_s, 12)
        c.find_source_neighbors(20)
        c.calculate_source_covariances(REG_PLANE)
        r = c.align()
        b.record(st)
        torch.cuda.synchronize()
        return a.elapsed_time(b), r

    def evaluation_ms(c, reps=10):
        st = torch.cuda.ExternalStream(c.stream(), device=dev)
        T = np.eye(4)
        c.linearize(T)
        torch.cuda.synchronize()
        D.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        for _ in range(reps):
            out = c.linearize(T)
        b.record(st)
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps, out

    rec = {"workload": "C4: synthetic 1M-pt pair (seeds 44/45), res 0.5, k=20 PLANE, LM defaults", "n_target": n_t, "n_source": n_s}
    c = Core(local_rank)
    c.set_resolution(0.5)
    out = {}
    for method in ("DIRECT27", "DIRECT1"):
        c.set_neighbor_search_method(method)
        for _ in range(2):
            registration(c)
        ts = [registration(c) for _ in range(3)]
        ms_reg = float(np.median([t for t, _ in ts]))
        res = ts[-1][1]
        ms_eval, (e_full, H_full, b_full) = evaluation_ms(c)
        c.set_profiling(True)
        for _ in range(5):
            c.linearize(np.eye(4))
        prof = c.get_profile()
        c.set_profiling(False)
        kern_ms = prof["linearize"][0] / max(prof["linearize"][1], 1)
        V, B = c.num_voxels(), c.num_buckets()
        alg = 52.0 * n_s + 52.0 * V + 16.0 * B
        ms_reg, ms_eval, kern_ms = D.max_over_ranks([ms_reg, ms_eval, kern_ms], device=dev)
        out[method] = {"ms_per_registration": ms_reg, "ms_per_evaluation_host_driven": ms_eval, "evaluation_kernel_ms": kern_ms, "num_voxels": V, "num_buckets": B,
                       "iterations": int(res.nr_iterations) + 1, "evaluations": int(res.n_linearize + res.n_compute_error), "converged": bool(res.converged),
                       "roofline": {"bound": "hbm", "kernel": "k_linearize<%s> (one LM evaluation of 1M source points)" % method, "algorithmic_bytes_per_launch": alg,
                                    "achieved": alg / (kern_ms * 1e-3) / 1e9, "peak": peak_gbs, "unit": "GB/s", "frac": alg / (kern_ms * 1e-3) / 1e9 / peak_gbs},
                       "_unsharded": (e_full, H_full, b_full, pose_from_c(res.T))}
        note("c4 %s: %.3f ms/registration, evaluation kernel %.1f us" % (method, ms_reg, 1e3 * kern_ms))
    # stage times of one registration (CUDA events around every launch)
    c.set_neighbor_search_method("DIRECT27")
    c.set_profiling(True)
    registration(c)
    prof = c.get_profile()
    c.set_profiling(False)
    rec["stage_ms_direct27"] = {k: v[0] for k, v in prof.items() if v[1]}
    if world > 1:
        sh = {}
        c2 = Core(local_rank)
        c2.set_resolution(0.5)
        # (host-driven LM loop with the speculative evaluation, as on one GPU: the device-resident chain -- no host round trip per
        # evaluation, but no speculation either -- measured 4.04 ms against 3.83 ms per sharded registration on 2 GPUs)
        lo, hi = D.setup_source_sharding(c2, n_s, max_points=max(n_s, n_t))
        for method in ("DIRECT27", "DIRECT1"):
            c2.set_neighbor_search_method(method)
            for _ in range(2):
                registration(c2)
            ts = [registration(c2) for _ in range(3)]
            ms_reg = float(np.median([t for t, _ in ts]))
            res = ts[-1][1]
            ms_eval, (e_sh, H_sh, b_sh) = evaluation_ms(c2)
            ms_reg, ms_eval = D.max_over_ranks([ms_reg, ms_eval], device=dev)
            e_full, H_full, b_full, T_full = out[method]["_unsharded"]
            T_sh = pose_from_c(res.T)
            sums = D.max_over_ranks([float(H_sh.sum()), -float(H_sh.sum()), float(T_sh.sum()), -float(T_sh.sum())], device=dev)
            sh[method] = {"ms_per_registration": ms_reg, "ms_per_evaluation_host_driven": ms_eval,
                          "speedup_vs_1": out[method]["ms_per_registration"] / ms_reg, "strong_scaling_efficiency": out[method]["ms_per_registration"] / ms_reg / world,
                          "evaluation_speedup_vs_1": out[method]["ms_per_evaluation_host_driven"] / ms_eval,
                          "H_rel_diff_vs_unsharded": float(np.abs(H_sh - H_full).max() / np.abs(H_full).max()),
                          "pose_abs_diff_vs_unsharded": float(np.abs(T_sh - T_full).max()),
                          "ranks_bit_identical": bool(sums[0] == -sums[1] and sums[2] == -sums[3]), "iterations": int(res.nr_iterations) + 1,
                          "converged": bool(res.converged)}
            note("c4 sharded x%d %s: %.3f ms/registration (x%.2f)" % (world, method, ms_reg, sh[method]["speedup_vs_1"]))
        err = int(D.max_over_ranks([float(c2.comm_error())], device=dev)[0])
        D.barrier()
        c2.comm_shutdown()
        c2.close()
        rec["sharded"] = dict(sh, n_gpus=world, comm_error=err, source_slice_of_rank0=[int(lo), int(hi)],
                              what="stage 1 (k-NN queries + covariances: peer stores into every rank's arrays) and stage 3 (evaluation: 28 sums per evaluation exchanged inside "
                                   "the kernel through NVLink peer mailboxes) sharded; k-NN grid build and voxel map replicated")
    for m in out.values():
        m.pop("_unsharded")
    rec.update(out)
    c.close()
    return rec


def write_outputs(out_dir, arrays, aligned_budget=16 << 20):
    """--dump-outputs: every array as out_dir/<name>.npy; the aligned clouds above `aligned_budget` bytes as a fixed, seeded sample of
    rows (the same rows for every stream) so that the files stay small at the 1M-point workloads."""
    os.makedirs(out_dir, exist_ok=True)
    a = arrays.get("e2e_aligned")
    if a is not None and a.nbytes > aligned_budget:
        n = a.shape[1]
        rows = np.sort(np.random.default_rng(0).choice(n, size=aligned_budget // (a.shape[0] * 12), replace=False))
        arrays["e2e_aligned"], arrays["e2e_aligned_rows"] = a[:, rows], rows.astype(np.float64)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), v)


# -------------------------------------------------------------------------------------------------------- GPU arm
def main():
    # stdout carries exactly one JSON line: route everything else that writes to fd 1 (NCCL's version banner, library
    # chatter) to stderr and keep a private handle on the real stdout for the result.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    # a run that stops making progress leaves the Python stacks of all threads on stderr every 5 minutes
    import faulthandler

    faulthandler.dump_traceback_later(300, repeat=True, file=sys.stderr)
    print("[bench] start", file=sys.stderr, flush=True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--streams", type=int, default=8,
                    help="concurrent registration streams per GPU (host thread + handle each); the same at every N (8 reach 98 %% of the 16-stream rate and "
                         "leave the host cores of a NUMA node to the ranks that share it)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="skip the 1M-point sub-record (config 4: evaluation roofline at N=1, sharded registration at N>1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (see the module docstring)")
    ap.add_argument("--e2e-impl", default="class", choices=["class", "batch"],
                    help="end-to-end arm: the FastVGICPCuda class from S Python threads (default, verified), or one vgicp_batch_register C call per timed region "
                         "(include/vgicp_batch_b200.h; not yet verified on hardware)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    w = load_workload(args.workload)

    if args.impl == "reference":
        run_reference_arm(args, w, rank, world)
        return

    print("[bench] importing torch (the first import on a fresh box pages the image in and can take minutes)", file=sys.stderr, flush=True)
    import torch

    print("[bench] torch imported", file=sys.stderr, flush=True)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    from fast_gicp_b200 import FastVGICPCuda, NDTCuda
    from fast_gicp_b200 import distributed as D
    from fast_gicp_b200.core import REG_PLANE, Core, pose_from_c

    D.init("nccl", dev)  # one rank per GPU; used for the barrier and the max-over-ranks of the device time only
    placement = pin_rank_threads(torch, local_rank, world)

    def barrier():
        D.barrier(cuda=True)

    tgt, src = w["target"], w["source"]
    n_t, n_s = len(tgt), len(src)
    K, W = args.steps, args.warmup
    S = max(args.streams, 1)
    _t0 = time.perf_counter()

    def note(msg):
        if rank == 0:
            print("[bench %7.1fs] %s" % (time.perf_counter() - _t0, msg), file=sys.stderr, flush=True)

    # ---- input pool: P distinct pairs (the workload pair under random rigid motions), P * pair bytes > L2 (126 MB), so a
    # pair has left the L2 by the time a stream comes back to it.  Resident copy for `value`, pinned host copy for `e2e`.
    pair_bytes = (n_t + n_s) * 12
    P = max(2 * S, int(np.ceil(160e6 / pair_bytes)))
    rng = np.random.default_rng(1234 + rank)
    tgt0 = torch.from_numpy(tgt).to(dev)
    src0 = torch.from_numpy(src).to(dev)
    pool_t = torch.empty((P, n_t, 3), dtype=torch.float32, device=dev)
    pool_s = torch.empty((P, n_s, 3), dtype=torch.float32, device=dev)
    for i in range(P):
        yaw = rng.uniform(-0.05, 0.05) if i else 0.0
        R = torch.tensor([[np.cos(yaw), -np.sin(yaw), 0.0], [np.sin(yaw), np.cos(yaw), 0.0], [0.0, 0.0, 1.0]], dtype=torch.float32, device=dev)
        t = torch.tensor(rng.uniform(-0.5, 0.5, size=3) * (1.0 if i else 0.0), dtype=torch.float32, device=dev)
        pool_t[i] = tgt0 @ R.T + t
        pool_s[i] = src0 @ R.T + t
    pool_t_h = torch.empty((P, n_t, 3), dtype=torch.float32).pin_memory()
    pool_s_h = torch.empty((P, n_s, 3), dtype=torch.float32).pin_memory()
    pool_t_h.copy_(pool_t)
    pool_s_h.copy_(pool_s)
    pool_t_np, pool_s_np = pool_t_h.numpy(), pool_s_h.numpy()
    aligned_h = [torch.empty((n_s, 3), dtype=torch.float32).pin_memory() for _ in range(S)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2 (single-stream latency pass)
    torch.cuda.synchronize()

    import threading

    note("input pool ready (%d pairs)" % P)
    ndt = w.get("problem") == "ndt_d2d"
    cores = [Core(local_rank) for _ in range(S)]
    regs = [(NDTCuda if ndt else FastVGICPCuda)(local_rank) for _ in range(S)]
    for r in regs:
        if ndt:
            r.vgicp_cuda_ = r.ndt_cuda_  # same accessor below
    for c in cores:
        if ndt:
            c.set_problem(2)
    # latency launch shapes + results through mapped host memory on every stream: measured faster than the throughput hint even at 16
    # handles per GPU (7.1k vs 6.7k registrations/s) since the evaluation kernel compacts its hits (scripts/exp_concurrency.py)
    hint = 0
    for c in cores:
        c.set_resolution(w["res"])
        c.set_neighbor_search_method(w["method"])
        c.set_execution_hint(hint)
    for r in regs:
        r.setResolution(w["res"])
        r.voxel_resolution_ = w["res"]
        r.setNeighborSearchMethod(w["method"], 0.0)
        r.vgicp_cuda_.set_execution_hint(hint)
    core = cores[0]
    streams = [torch.cuda.ExternalStream(c.stream(), device=dev) for c in cores]
    e2e_streams = [torch.cuda.ExternalStream(r.vgicp_cuda_.stream(), device=dev) for r in regs]
    stream = streams[0]
    tp, sp = pool_t.data_ptr(), pool_s.data_ptr()

    def step_resident(ci=0, pi=0):
        """One registration with both clouds resident in HBM: the C-ABI call sequence of setInputTarget + setInputSource + align."""
        c = cores[ci]
        if ndt:  # NDTCuda: setInputTarget + setInputSource + align (voxel maps from the raw points inside align)
            c.set_cloud_device("target", tp + pi * n_t * 12, n_t, 12)
            c.set_cloud_device("source", sp + pi * n_s * 12, n_s, 12)
            c.ndt_create_voxelmaps()
            return c.align()
        # vgicp_register = clear + setInputTarget (kNN, covariances, voxel map) + setInputSource (kNN, covariances) + align in one
        # C call: the body of the reference's benchmark loop (src/align.cpp:72-81), no Python between the stages
        return c.register_raw(tp + pi * n_t * 12, n_t, sp + pi * n_s * 12, n_s, 12, True, 20, REG_PLANE)

    def step_e2e(ci=0, pi=0):
        """The same through the reference-facing class, host (pinned) buffers in, aligned cloud + pose out (align.cpp:72-81)."""
        r = regs[ci]
        r.clearTarget()
        r.clearSource()
        r.setInputTarget(pool_t_np[pi])
        r.setInputSource(pool_s_np[pi])
        return r.align(aligned_out=aligned_h[ci].numpy())

    def run_streams(step_fn, stream_list, steps):
        """`steps` registrations on each of the S streams (one host thread + one handle per stream), distinct pairs from the
        pool; returns (device time from the common start event to the last stream's end event [ms], last result of every stream)."""
        start = torch.cuda.Event(enable_timing=True)
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(S)]
        out = [None] * S
        gate = threading.Barrier(S + 1)

        def work(ci):
            gate.wait()
            for j in range(steps):
                out[ci] = step_fn(ci, (ci + j * S) % P)
            ends[ci].record(stream_list[ci])

        th = [threading.Thread(target=work, args=(ci,)) for ci in range(S)]
        for t_ in th:
            t_.start()
        torch.cuda.synchronize()
        start.record(torch.cuda.current_stream())
        torch.cuda.current_stream().synchronize()
        gate.wait()
        for t_ in th:
            t_.join()
        torch.cuda.synchronize()
        return max(start.elapsed_time(e) for e in ends), out

    # ---- value: resident inputs, S concurrent streams
    note("handles ready")
    run_streams(step_resident, streams, W)
    note("warm-up done")
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    l0 = sum(c.launch_count() for c in cores)
    t_wall0 = time.perf_counter()
    total_ms, last = run_streams(step_resident, streams, K)
    barrier()
    wall_s = time.perf_counter() - t_wall0
    launches = sum(c.launch_count() for c in cores) - l0
    res = last[0]
    dump = {}
    if args.dump_outputs:
        dump["pose"] = np.stack([pose_from_c(r.T) for r in last])
        dump["hessian"] = np.stack([np.array(r.H).reshape(6, 6).T for r in last])

    # ---- e2e: host buffers through the reference-facing class, S concurrent streams
    note("value arm done")
    e2e_api = "FastVGICPCuda.setInputTarget/setInputSource/align (pinned host buffers, aligned cloud + pose read back)"
    if args.e2e_impl == "batch" and not ndt:
        # one C call for all S*K registrations: a pool of S handles + worker threads inside libvgicp_batch_b200.so, pinned host buffers in,
        # aligned clouds + poses out; device time = events on the current stream around the (blocking) call
        from fast_gicp_b200.batch import BatchRegistration

        pool = BatchRegistration(local_rank, S)
        pool.configure(w["res"], w["method"])
        aligned_all = [torch.empty((n_s, 3), dtype=torch.float32).pin_memory().numpy() for _ in range(S * max(K, W))]

        def run_batch(steps):
            idx = [(ci + j * S) % P for j in range(steps) for ci in range(S)]
            call = pool.prepare([pool_t_np[i] for i in idx], [pool_s_np[i] for i in idx], aligned_all[: len(idx)])
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            ev0.record()
            res_b = call(20, REG_PLANE)
            ev1.record()
            torch.cuda.synchronize()
            return ev0.elapsed_time(ev1), res_b

        run_batch(W)
        barrier()
        total_ms_e2e, last_e2e = run_batch(K)
        barrier()
        T_e2e = pose_from_c(last_e2e[0].T)
        if args.dump_outputs:  # the last S registrations of the call are the last step's
            dump["e2e_pose"] = np.stack([pose_from_c(r.T) for r in last_e2e[-S:]])
            dump["e2e_aligned"] = np.stack(aligned_all[S * K - S:S * K])
        launches_e2e = int(launches)  # the pool's handles are internal: same launches per registration as the resident arm
        e2e_api = "vgicp_batch_register (one C call for all registrations of the timed region; pinned host buffers, aligned clouds + poses read back)"
    else:
        run_streams(step_e2e, e2e_streams, W)
        barrier()
        l1 = sum(r.vgicp_cuda_.launch_count() for r in regs)
        total_ms_e2e, last_e2e = run_streams(step_e2e, e2e_streams, K)
        barrier()
        T_e2e = last_e2e[0]
        if args.dump_outputs:
            dump["e2e_pose"] = np.stack(last_e2e).astype(np.float64)
            dump["e2e_aligned"] = np.stack([a.numpy() for a in aligned_h])
        launches_e2e = sum(r.vgicp_cuda_.launch_count() for r in regs) - l1
    clocks = sampler.stop() if sampler else None

    # ---- single-stream latency (the reference's sequential protocol), L2 flushed between registrations
    note("e2e arm done")
    cores[0].set_execution_hint(0)
    regs[0].vgicp_cuda_.set_execution_hint(0)
    lat = []
    for j in range(W + min(K, 30)):
        flush.zero_()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        step_resident(0, j % P)
        b.record(stream)
        torch.cuda.synchronize()
        if j >= W:
            lat.append(a.elapsed_time(b))
    lat_e2e = []
    for j in range(W + min(K, 30)):
        flush.zero_()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(e2e_streams[0])
        step_e2e(0, j % P)
        b.record(e2e_streams[0])
        torch.cuda.synchronize()
        if j >= W:
            lat_e2e.append(a.elapsed_time(b))

    note("single-stream pass done")
    # ---- max over ranks
    total_ms, total_ms_e2e = D.max_over_ranks([total_ms, total_ms_e2e], device=dev)

    # ---- the same pair in the reference's published configurations (README.md:129-134 rows are DIRECT1: align.cpp never sets a
    # neighbour method; :133-134 is the RBF-covariance mode), N = 1 only: sub-records, not the headline
    extras = {}
    if args.workload == "c2" and world == 1 and not ndt:
        def timed_single(fn, reps=20):
            ts = []
            for j in range(3 + reps):
                flush.zero_()
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                fn(j % P)
                b.record(stream)
                torch.cuda.synchronize()
                if j >= 3:
                    ts.append(a.elapsed_time(b))
            return float(np.mean(ts))

        for c in cores:
            c.set_neighbor_search_method("DIRECT1")
        run_streams(step_resident, streams, W)
        ms_d1, _ = run_streams(step_resident, streams, min(K, 20))
        extras["c2_direct1"] = {"value": S * min(K, 20) / (ms_d1 * 1e-3), "unit": UNIT, "streams_per_gpu": S,
                                "single_stream_ms": timed_single(lambda pi: step_resident(0, pi)),
                                "published_reference": "vgicp_cuda 68.9 registrations/s (100x protocol, kd-tree kNN on the CPU, RTX 2080 Ti + i9-9900K, README.md:129-130)"}

        def step_rbf(pi):  # NearestNeighborMethod::GPU_RBF_KERNEL: covariances from the kernel-weighted neighbourhood, no kNN
            c = cores[0]
            c.set_cloud_device("target", tp + pi * n_t * 12, n_t, 12)
            c.calculate_target_covariances_rbf(REG_PLANE)
            c.create_target_voxelmap()
            c.set_cloud_device("source", sp + pi * n_s * 12, n_s, 12)
            c.calculate_source_covariances_rbf(REG_PLANE)
            return c.align()

        cores[0].set_kernel_params(0.5, 3.0)  # fast_vgicp_cuda_impl.hpp:31
        ms_rbf = timed_single(step_rbf)
        cores[0].set_profiling(True)
        for j in range(5):
            step_rbf(j)
        pr = cores[0].get_profile()
        cores[0].set_profiling(False)
        extras["c2_direct1_rbf"] = {"single_stream_ms": ms_rbf, "registrations_per_s": 1e3 / ms_rbf, "covariance_ms_per_cloud": pr["covariance"][0] / max(pr["covariance"][1], 1),
                                    "published_reference": "vgicp_cuda (GPU RBF kernel) 169.3 registrations/s (README.md:133-134)"}
        for c in cores:
            c.set_neighbor_search_method(w["method"])
        note("DIRECT1 / RBF sub-records done")

    # ---- per-kernel profile (separate pass, events around every launch) -> roofline of the dominant kernel
    core.set_profiling(True)
    for j in range(min(K, 20)):
        flush.zero_()
        torch.cuda.synchronize()
        step_resident(0, j % P)
    prof = core.get_profile()
    core.set_profiling(False)
    n_prof = min(K, 20)
    per_kernel = {k: {"ms_per_step": v[0] / n_prof, "launches_per_step": v[1] / n_prof} for k, v in prof.items() if v[1]}

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak_gbs, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak_gbs, peak_src = 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"
    V, B = core.num_voxels(), core.num_buckets()
    # ---- config 4 (all ranks take part: sharded over the ranks when there are several)
    c4 = None
    if args.workload == "c2" and not args.no_c4:
        for c_ in cores[1:]:
            c_.close()
        del pool_t, pool_s, flush
        torch.cuda.empty_cache()
        try:
            c4 = c4_record(torch, dev, local_rank, rank, world, peak_gbs, note)
        except Exception as e:  # noqa: BLE001
            c4 = {"error": repr(e)}
        note("c4 record done")

    if rank != 0:
        D.finalize()
        return
    # algorithmic bytes per launch, SURVEY.md 8(d)
    if ndt:
        METRIC_NAME = "registrations/sec (NDT D2D, KITTI-shaped pairs)"
    else:
        METRIC_NAME = METRIC
    alg_bytes = {
        "knn": 52.0 * 0.5 * (n_t + n_s),                    # stage 1 (kNN+cov+reg) 52 B/pt, one cloud per launch
        "covariance": 52.0 * 0.5 * (n_t + n_s),
        "voxelmap_build": 52.0 * n_t + 52.0 * V + 16.0 * B,  # stage 2, whole build
        "linearize": 52.0 * n_s + 52.0 * V + 16.0 * B,       # stage 3, one LM evaluation
        "compute_error": 52.0 * n_s + 52.0 * V + 16.0 * B,
    }
    # kernel groups as they appear in the ncu launch list: the evaluation kernel k_linearize<MODE,WANT_H,G> (linearize and
    # error-only calls are the same template), the k-NN stage (Morton grid build + k_knn_search + k_knn_deferred), ...
    groups = {"evaluate (k_linearize, H and error-only)": ["linearize", "compute_error"], "knn stage (k_grid_* + k_sort_pass + k_knn_search + k_knn_deferred)": ["knn"],
              "covariance (k_covariance_knn)": ["covariance"], "voxelmap_build (table, ids, sort, ordered per-voxel sums)": ["voxelmap_build"]}
    total_kernel_ms = sum(v["ms_per_step"] for v in per_kernel.values()) or 1.0

    def group_roofline(gname):
        cats = [c for c in groups[gname] if c in per_kernel]
        ms = sum(per_kernel[c]["ms_per_step"] for c in cats)
        launches_g = 1.0 if "voxelmap" in gname else sum(per_kernel[c]["launches_per_step"] for c in cats)  # one map build per registration
        avg_ms = ms / max(launches_g, 1e-9)
        ab = alg_bytes[cats[0]]
        ach = ab / (avg_ms * 1e-3) / 1e9
        traffic = None  # ncu dram__bytes per launch, written by scripts/make_traffic.sh; quoted only while the kernels are the ones it measured
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            vals = [tj[c] for c in cats if c in tj]
            if tj.get("source_hash") == source_hash() and vals:
                traffic = float(np.mean(vals))
        return {"bound": "hbm", "kernel": gname, "achieved": ach, "peak": peak_gbs, "unit": "GB/s", "frac": ach / peak_gbs, "traffic": traffic, "peak_source": peak_src,
                "avg_launch_ms": avg_ms, "algorithmic_bytes_per_launch": ab, "kernel_share_of_step": ms / total_kernel_ms}

    present = [g for g in groups if any(c in per_kernel for c in groups[g])]
    rl = {g: group_roofline(g) for g in present}
    dom = max(present, key=lambda g: rl[g]["kernel_share_of_step"])
    roofline = rl[dom]
    roofline["note"] = ("at ~17k points every kernel is latency/issue-bound (one evaluation moves ~1 MB = 0.17 us at the HBM peak); the fraction is reported as the "
                        "contract asks, the 1M-point numbers are in profiles/README.md")
    roofline_other = {g: {k: rl[g][k] for k in ("achieved", "frac", "avg_launch_ms", "kernel_share_of_step", "algorithmic_bytes_per_launch", "traffic")} for g in present if g != dom}

    note("profile pass done")
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        # in a clean subprocess (own OpenMP runtime, no CUDA threads around), passive waiting, hard time limit
        env = dict(os.environ, OMP_WAIT_POLICY="PASSIVE")
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "60", "--warmup", "2", "--workload", args.workload],
                                 capture_output=True, text=True, timeout=150, env=env)
            ref = json.loads(out.stdout.strip().splitlines()[-1])
            cpu_baseline = ref["cpu_baseline"]
            cpu_baseline["host_cores"] = os.cpu_count()
        except Exception as e:  # noqa: BLE001
            cpu_baseline = {"value": None, "unit": UNIT, "cores": None, "kind": "port", "sample": "failed: %r" % (e,)}
    note("cpu baseline done")
    T_val = pose_from_c(res.T)
    h2d = (n_t + n_s) * 12
    d2h = n_s * 12 + 16 * 4 + (res.n_linearize * 43 + res.n_compute_error) * 8
    line = {
        "metric": METRIC_NAME, "value": world * S * K / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": w["data"],
        "config": {"workload": w["name"], "protocol": "align.cpp 100times (covariances recomputed every registration)", "step": "one registration on each of the %d concurrent streams of a GPU (one host thread + one handle per stream)" % S,
                   "streams_per_gpu": S, "cuda_device_max_connections": int(os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS", "8")), "registrations_per_step": S * world, "execution_hint": "throughput" if hint else "latency",
                   "l2": "inputs larger than L2: each registration takes the next of %d distinct pairs (%.0f MB pool)" % (P, P * pair_bytes / 1e6),
                   "parallelism": "replicas x%d" % world, "n_target": n_t, "n_source": n_s, "num_voxels": V, "num_buckets": B,
                   "lm_iterations": int(res.nr_iterations) + 1, "evaluations": int(res.n_linearize + res.n_compute_error), "converged": bool(res.converged)},
        "e2e": {"value": world * S * K / (total_ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d * S, "d2h_bytes_per_step": d2h * S, "ms_per_step": total_ms_e2e / K,
                "api": e2e_api},
        "gpu_launches": int(launches), "gpu_launches_e2e": int(launches_e2e),
        "roofline": roofline, "roofline_other_kernels": roofline_other, "cpu_baseline": cpu_baseline, "clocks": clocks, "per_kernel": per_kernel,
        "single_stream": {"ms_per_registration": float(np.mean(lat)), "registrations_per_s": 1e3 / float(np.mean(lat)),
                          "e2e_ms_per_registration": float(np.mean(lat_e2e)), "e2e_registrations_per_s": 1e3 / float(np.mean(lat_e2e)),
                          "l2": "flushed between registrations (256 MiB memset)", "protocol": "sequential, as src/align.cpp:72-81"},
        "wall_ms_per_step": 1e3 * wall_s / K, "host_placement": placement, "c4": c4, "published_configurations": extras,
        "pose_check": {"translation": [float(x) for x in T_val[:3, 3]], "e2e_vs_resident_max_abs": float(np.abs(np.asarray(T_e2e, dtype=np.float64) - T_val).max())},
    }
    if args.dump_outputs:
        dump["counters"] = np.array([[r.nr_iterations, r.converged, r.n_linearize, r.n_compute_error, r.lm_failed] for r in last], dtype=np.float64)
        write_outputs(args.dump_outputs, dump)
    print(json.dumps(line), file=_REAL_STDOUT, flush=True)
    D.finalize()


if __name__ == "__main__":
    main()
