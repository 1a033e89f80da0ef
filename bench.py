#!/usr/bin/env python
"""bench.py — NDT scan-matches/sec on the workload BASELINE.json's metric is quoted on.

Workload (N = 1 and per rank for N > 1): BASELINE.json configs[1], "scan-to-map NDT align, 1080-beam scans vs
200 x 200 m map at 0.25 m cells". One step = one batched align pass over `--scans` synthetic 1080-beam scans
(SURVEY.md 8(d) generator) against the same map; every scan runs the full Levenberg-Marquardt loop of SPEC.md 5.

  value   whole-job matches/s with scans, offsets and initial poses already resident in HBM
  e2e     the same through the host-buffer C-ABI call (ndt2d_align_batch / _ranges): pinned host -> device copy
          of the step's scans, kernel, device -> host copy of the results, all inside the timed region
  roofline  Newton-step evaluations x algorithmic bytes (N*(8+32K)+92, BASELINE.md section 5) / kernel time,
          against the measured HBM copy bandwidth (MEASURED_PEAKS.json). It is a gather-traffic convention:
          the cell table is L2-resident, so the fraction is not DRAM utilisation (DESIGN.md).
  cpu_baseline  the CPU spec oracle (a port of SPEC.md; the reference mount holds no source) on the host cores

--impl reference times that same CPU oracle as the reference arm (the reference's own matcher does not exist
in /root/reference; see BASELINE.md). Multi-GPU: independent scans are sharded per rank, no data-path collective.

The default run (`--workload scan2map`, what the driver launches at N = 1, 2, 4, 8) adds these legs to the same JSON line
(`--legs none` skips them):
  sweep     configs[3]: 1 M pose hypotheses x one 1080-pt scan, sharded over the N ranks (strong scaling), best-hypothesis
            combine by peer-memory stores from the arg-max kernel and, beside it, by an NCCL all-gather; 48 sharded queries
            with cross-shard ties are checked against the unsharded sweep on every rank - a mismatch makes the bench exit 3
  pyramid   configs[2]: 2.0/1.0/0.5 m pyramid, 10 000 scans in total sharded over the ranks, prior error 0.2 m / 3 deg
  prior2    configs[1] again with the 0.2 m / 3 deg prior (matches/s depends on the prior through the iteration count)
  odometry  batched scan-to-scan (ndt2d_align_pairs): 16 384 consecutive scans per GPU, pair k = (scan k-1 -> scan k), 0.5 m cells
  dense     configs[1] in a cluttered world whose map has > 300 k valid cells (the default room has 14 k)
  config0   configs[0]: one 360-beam scan-to-scan align at 0.5 m cells, CPU oracle on one thread vs ndt2d_align latency
  config4   configs[4], the front end: examples/slam_frontend.cpp (GPU odometry + loop closure -> g2o pose graph), its own figures
  precision distance of the GPU results from an independent f64 NDT (oracle/f64ref.py) at north_star's tolerances
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the bench writes nothing into the tree (which may be read-only)

METRIC = "NDT scan-matches/sec (1080-pt 2D scans)"
UNIT = "matches/s"
DUMP_BUDGET = 64 << 20              # --dump-outputs: bytes in all, over every rank
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 10; 50 for --workload sweep, whose steps are 0.3-2 ms)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="scan2map", choices=["scan2map", "pyramid", "sweep", "build", "newton", "odometry"],
                    help="scan2map: BASELINE configs[1] (default, the metric's config); pyramid: configs[2] (2.0/1.0/0.5 m, "
                         "10k scans, 0.2 m / 3 deg prior error); sweep: configs[3] (1M hypotheses x one 1080-pt scan)")
    ap.add_argument("--hyps", type=int, default=1000000, help="sweep: total hypotheses (sharded across GPUs)")
    ap.add_argument("--combine", default="p2p", choices=["p2p", "nccl"],
                    help="sweep on N > 1 GPUs: best-hypothesis combine by peer-memory stores from the arg-max kernel (p2p) "
                         "or by an NCCL all-gather on a side stream (nccl)")
    ap.add_argument("--scans", type=int, default=None, help="scans per step per GPU (65536 x 1080 x 8 B = 566 MB, far above the 126 MB L2)")
    ap.add_argument("--map-scans", type=int, default=2048, help="scans fused into the target map")
    ap.add_argument("--res", type=float, nargs="+", default=None)
    ap.add_argument("--overlap", type=int, default=0)
    ap.add_argument("--perturb", type=float, nargs=2, default=None, help="initial guess error: metres, degrees")
    ap.add_argument("--input", default="ranges_f32", choices=["xy", "ranges_f32", "ranges_u16"],
                    help="host input of the e2e leg: LaserScan ranges (what the sensor delivers; f32, SPEC.md section 8) or already "
                         "converted float2 points; every format is timed and listed under e2e.by_input. The CPU arms always get points.")
    ap.add_argument("--cpu-sample", type=int, default=0, help="scans in the cpu_baseline sample (0: auto, about 10-20 s)")
    ap.add_argument("--ref-scans", type=int, default=0, help="scans per step of the reference arm (0: auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--legs", default="all", help="scan2map only: extra legs in the same JSON line: all | none | comma list of "
                                                  "sweep,pyramid,prior2,odometry,dense,config0,config4,precision")
    ap.add_argument("--world", default="room", choices=["room", "dense"],
                    help="synthetic world of the scan2map workload: the SURVEY 8(d) room (14 k valid map cells) or the cluttered dense world (> 300 k)")
    ap.add_argument("--relay", default="auto", choices=["auto", "off"],
                    help="e2e on several GPUs: auto = ranks whose host-to-device rate is lower than a peer's relay a share of their input "
                         "through that peer's GPU (ndt2d_set_upload_relay); off = every rank uses its own PCIe link only")
    ap.add_argument("--pinned", default="default", choices=["default", "wc"],
                    help="e2e input buffer: ordinary pinned memory, or write-combined pinned memory (ndt2d_host_alloc_flags)")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to the NUMA node of its GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="scan2map and the reference arm: after the timed steps, write the result records of the last step as "
                         "DIR/<field>.npy (float64; at most 64 MB, a fixed seeded sample of the scans above that), so that two builds "
                         "can be compared output for output")
    a = ap.parse_args()
    if (a.steps is not None and a.steps < 1) or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl == "native" and a.workload != "scan2map":
        ap.error("--dump-outputs: only the scan2map workload and the reference arm write their outputs")
    dflt = {"scan2map": (65536, [0.25], [0.03, 0.3]), "pyramid": (10000, [2.0, 1.0, 0.5], [0.2, 3.0]), "sweep": (1, [0.25], [0.0, 0.0]),
            "build": (1, [0.25], [0.0, 0.0]), "newton": (1, [0.25], [0.0, 0.0]),
            "odometry": (16384, [0.5], [0.02, 0.2])}[a.workload]
    a.scans = a.scans or dflt[0]
    if a.steps is None:
        a.steps = 50 if a.workload == "sweep" else 10
    a.res = a.res or dflt[1]
    a.perturb = a.perturb or dflt[2]
    legs = ["sweep", "pyramid", "prior2", "odometry", "dense", "config0", "config4", "precision"]
    a.legs = legs if a.legs == "all" else [] if a.legs == "none" else [x for x in a.legs.split(",") if x]
    if a.workload != "scan2map" or a.overlap or a.world != "room" or a.res != [0.25]:
        a.legs = []          # the legs belong to the default configuration
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks and throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_workload(args, rank, with_map=True, count=None, dense=False):
    """Synthetic scans for this rank (distinct trajectory slots per rank), the shared map, and initial guesses.
    `count` < args.scans takes the first scans of the same workload (bounded CPU samples). dense: the cluttered world
    (synth.set_world(dense=True) must be in force); its map is the surveyed box edges, not a lidar map."""
    from gtsam_ndt_b200 import synth
    world = max(1, args.gpus)
    traj = args.scans * world
    sc = synth.SCAN_1080
    count = count or args.scans
    ranges, poses = synth.scans(count, traj_len=traj, first=rank, step=world, nboxes=synth.DENSE_NBOXES if dense else synth.NBOXES, **sc)
    pert = synth.uniform3(count, first=rank * args.scans) * np.array([args.perturb[0], args.perturb[0], math.radians(args.perturb[1])])
    init = poses + pert
    map_xy = None
    if with_map:
        map_xy = synth.dense_map() if dense else synth.make_map(args.map_scans, traj_len=args.map_scans, **sc)
    return ranges, poses, init, map_xy


def to_points(ranges):
    """SPEC 8 conversion on the host; all 1080 beams return in this world, so the batch is rectangular."""
    from gtsam_ndt_b200 import synth
    sc = synth.SCAN_1080
    cb, sb = synth.beam_table(sc["nbeams"], sc["angle_min"], sc["angle_inc"])
    assert np.all(ranges > 0)
    xy = np.stack([ranges * cb[None, :], ranges * sb[None, :]], axis=-1).astype(np.float32)
    offsets = np.arange(ranges.shape[0] + 1, dtype=np.int64) * ranges.shape[1]
    return xy.reshape(-1, 2), offsets


def dump_records(out_dir, res, rank=0, world=1):
    """--dump-outputs: every field of the result records (pose, score, grad, hessian, iterations, status, count) as
    out_dir/<field>.npy in float64, one row per scan; rank r of a multi-GPU job writes <field>_rank<r>.npy. When the
    records exceed this rank's share of DUMP_BUDGET, the same seeded sample of scans is written on every run, and
    index.npy holds the sampled scan indices."""
    fields = [f for f in res.dtype.names if f != "reserved"]
    row_bytes = 8 * (1 + sum(int(np.prod(res.dtype[f].shape)) for f in fields))
    rows = (DUMP_BUDGET // max(1, world) - 4096 * (len(fields) + 1)) // row_bytes
    arrays = {}
    if len(res) > rows:
        arrays["index"] = np.sort(np.random.default_rng(0).choice(len(res), rows, replace=False))
        res = res[arrays["index"]]
    arrays.update((f, res[f]) for f in fields)
    suffix = f"_rank{rank}" if world > 1 else ""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def ncu_traffic(kernel, args, scans):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu capture of this exact
    configuration (profiles/traffic.json); None when no capture matches."""
    try:
        tab = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        key = "%s/%s/scans=%d/res=%s/K=%d" % (kernel, args.workload, scans, "-".join(str(r) for r in args.res), 4 if args.overlap else 1)
        return tab.get(key, {}).get("dram_bytes")
    except Exception:
        return None


def gather_pipe(kernel_key, kernel_ms, clocks, sm_count):
    """The path's real ceiling next to the HBM figure: an SM's L1TEX data pipe takes one cycle per distinct 32 B sector of
    a gather (DESIGN.md section 5). Sector count per launch from the committed ncu capture of this configuration."""
    try:
        tab = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        sectors = tab[kernel_key]["l1tex_sectors"]
        mhz = (clocks or {}).get("sm_mhz") or 1965.0
        peak = sm_count * mhz * 1e6
        ach = sectors / (kernel_ms / 1e3)
        return {"sectors_per_launch": sectors, "achieved_sectors_per_s": ach, "peak_sectors_per_s": peak, "frac": ach / peak,
                "note": "l1tex__t_sectors_pipe_lsu_mem_global_op_ld from the ncu capture; peak = SMs x SM clock (one sector per cycle per SM)"}
    except Exception:
        return None


def ncu_pipes(kernel_key):
    """Utilisation of the units that share the limit of this kernel, from the committed ncu capture of the configuration
    (static, like `traffic`; `commit` names the build): issue slots, FMA pipe, L1TEX data pipe, L2 hit rate."""
    try:
        e = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[kernel_key]
        out = {k: e[k] for k in ("issue_active_pct", "fma_pipe_cycles_active_pct", "l1tex_data_pipe_pct", "l2_hit_pct", "inst_executed") if k in e}
        out["commit"] = e.get("commit")
        out["source"] = e.get("source")
        return out
    except Exception:
        return None


def instruction_mix(kernel_key, kernel_ms, clocks, sm_count, evals, npts):
    """How close the point loop is to the speed of light of its own instruction mix. tools/mix_probe.py issues the loop's
    instruction counts from independent register chains (no memory, no dependencies): its cycles per body per scheduler are
    the floor any schedule of the mix has (`mix_floor_cycles`: classes grouped / interleaved). The loop's actual cycles per
    64-point step per scheduler = live kernel time x clock x schedulers x the loop's share of the kernel's PC samples / steps."""
    try:
        e = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[kernel_key]
        floor, share = e["mix_floor_cycles"], e["loop_sample_share"]
        mhz = (clocks or {}).get("sm_mhz") or 1965.0
        steps = evals * ((npts + 63) // 64)
        cyc = kernel_ms * 1e-3 * mhz * 1e6 * sm_count * 4 * share / steps
        return {"loop_cycles_per_step_per_scheduler": cyc, "mix_floor_cycles": floor, "frac_of_grouped_floor": floor[0] / cyc,
                "frac_of_interleaved_floor": floor[1] / cyc, "loop_sample_share": share,
                "note": "floor: profiles/r3n_mix_probe.txt (tools/mix_probe.py); share: profiles/r3k_k_align_loop_stalls.txt"}
    except Exception:
        return None


def ncu_traffic_sweep(args, hyps):
    try:
        tab = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        key = "k_eval_poses/sweep/hyps=%d/res=%s/K=%d" % (hyps, "-".join(str(r) for r in args.res), 4 if args.overlap else 1)
        return tab.get(key, {}).get("dram_bytes")
    except Exception:
        return None


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def eval_bytes(npts, K):
    return npts * (8 + 32 * K) + 12 + 80


def run_reference(args):
    """Reference arm: the CPU spec oracle (no upstream matcher exists in the mount), all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from gtsam_ndt_b200 import synth
    o = oracle.Oracle(args.res, overlap=args.overlap)
    o.set_grid(-100.0, -100.0, 200.0, 200.0)
    cores = host_cores()      # torchrun exports OMP_NUM_THREADS=1; the arm uses every core the process may run on
    nref = args.ref_scans or args.scans      # the native arm's batch (same config); ~1 s per step on 16 cores
    ranges, poses, init, map_xy = make_workload(args, 0, count=nref)
    o.set_target(map_xy)
    xy, off = to_points(ranges)
    for _ in range(args.warmup):
        o.align_batch(xy, off, init, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):         # the CPU arm gets already converted points: its polar-to-point conversion is not charged
        res = o.align_batch(xy, off, init, nthreads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_records(args.dump_outputs, res)
    v = nref * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64 point-to-cell geometry, f32 cell-local algebra, f64 sums and solver", "data": "synthetic",
            "config": workload_config(args, nref, extra={"world": args.world, "valid_map_cells": int((o.cells(len(args.res) - 1)[..., 7] != 0).sum())}),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{nref} scans x {args.steps} steps, CPU spec oracle (SPEC.md port; reference mount has no source), host input: float2 points (conversion from ranges not charged)"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "mean_iterations": float(res["iterations"].mean()), "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_config(args, scans, extra=None):
    K = 4 if args.overlap else 1
    name = {"scan2map": "configs[1]: scan-to-map NDT align", "pyramid": "configs[2]: multi-resolution NDT align (pyramid)",
            "sweep": "configs[3]"}[args.workload]
    c = {"workload": "%s, 1080-beam scans vs 200x200 m map at %s m cells (K=%d), batch of %d scans per GPU per step"
         % (name, "/".join(str(r) for r in args.res), K, scans),
         "scans_per_step_per_gpu": scans, "points_per_scan": 1080, "cell_res_m": list(args.res), "K": K,
         "map_points": args.map_scans * 1080, "init_error": {"trans_m": args.perturb[0], "rot_deg": args.perturb[1]},
         "l2": "per-step scan input %.0f MB > 126 MB L2 (no flush needed); the 200x200 m cell table is L2-resident by design"
               % (scans * 1080 * 8 / 1e6),
         "parallelism": "independent scans sharded per GPU, no collective"}
    if extra:
        c.update(extra)
    return c


class Ctx:
    """One rank of the bench: device, stream, process group (NCCL when world > 1) and the NUMA placement of the host side."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if self.world != max(1, args.gpus) and self.world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the NDT path has no CPU fallback (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.affinity0 = sorted(os.sched_getaffinity(0))
        from gtsam_ndt_b200 import synth
        synth.set_threads(max(1, len(self.affinity0) // self.world))   # torchrun exports OMP_NUM_THREADS=1: take this rank's share
        self.numa = {"bound": False, "note": "--no-numa"} if args.no_numa else bind_to_gpu_numa(self.local)
        if self.world > 1:
            # stdout carries exactly one JSON line: NCCL prints its version banner there when NCCL_DEBUG=VERSION/INFO is set, so
            # the descriptor points at stderr while the communicator is created (NCCL_DEBUG itself is left alone)
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=self.dev)
                t = torch.zeros(1, device=self.dev)
                dist.all_reduce(t)
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)
        self.stream = torch.cuda.current_stream()

    def sync_all(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        if self.world == 1:
            return [float(v) for v in vals]
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def sum_over_ranks(self, *vals):
        if self.world == 1:
            return [float(v) for v in vals]
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(v) for v in t]

    def gather_floats(self, v):
        if self.world == 1:
            return [float(v)]
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device=self.dev)
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(x) for x in out]

    def timed(self, fn, steps, warmup, drain=None):
        """W warm-up calls, then `steps` calls between CUDA events on the stream the kernels are launched on; barrier and
        synchronise on both sides; returns this rank's milliseconds for all the steps."""
        for _ in range(warmup):
            fn()
        if drain:
            drain()
        self.sync_all()
        e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for _ in range(steps):
            fn()
        if drain:
            drain()
        e1.record(self.stream)
        self.sync_all()
        return e0.elapsed_time(e1)

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def bind_to_gpu_numa(local):
    """Run this rank's host threads on the NUMA node its GPU hangs off, BEFORE any pinned buffer is allocated: the pages
    of a cudaHostAlloc are placed by first touch, so the copies then never cross the socket interconnect. Best effort:
    inside a cpuset that excludes that node nothing changes, and the line says so."""
    info = {"bound": False}
    try:
        import torch
        prop = torch.cuda.get_device_properties(local)
        if hasattr(prop, "pci_bus_id"):
            bdf = "%04x:%02x:%02x.0" % (prop.pci_domain_id, prop.pci_bus_id, prop.pci_device_id)
        else:       # older torch: ask the driver (the index is the CUDA ordinal only without CUDA_VISIBLE_DEVICES remapping)
            out = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.strip()
            bdf = out[-12:].lower()
        info["gpu_pci"] = bdf
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        info["gpu_numa_node"] = node
        allowed = set(os.sched_getaffinity(0))
        nodes = numa_nodes()
        info["host_numa_nodes"] = {str(k): len(v & allowed) for k, v in nodes.items()}
        if node < 0:
            # virtualised platforms report -1: find the node by measurement (pinned buffer first-touched on each node in turn)
            usable = {k: v & allowed for k, v in nodes.items() if v & allowed}
            if len(usable) < 2:
                info["note"] = "the platform reports no NUMA node for the GPU and the process can run on one node only"
                return info
            probe = {}
            for k, cpus_k in usable.items():
                os.sched_setaffinity(0, cpus_k)
                h = torch.empty(64 << 20, dtype=torch.uint8).pin_memory()
                h.zero_()
                d = torch.empty_like(h, device=torch.device("cuda", local))
                d.copy_(h, non_blocking=True)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(4):
                    d.copy_(h, non_blocking=True)
                e1.record()
                torch.cuda.synchronize()
                probe[k] = 4 * h.numel() / (e0.elapsed_time(e1) / 1e3) / 1e9
                del h, d
            os.sched_setaffinity(0, allowed)
            node = max(probe, key=probe.get)
            info["probe_h2d_gbs_by_node"] = {str(k): round(v, 1) for k, v in probe.items()}
            info["gpu_numa_node"] = node
            info["note"] = "node chosen by measured pinned-copy bandwidth (sysfs reports -1)"
        cpus = nodes.get(node, set())
        info["allowed_cpus"] = len(allowed)
        info["allowed_on_gpu_node"] = len(allowed & cpus)
        if allowed & cpus and (allowed & cpus) != allowed:
            os.sched_setaffinity(0, allowed & cpus)
            info["bound"] = True
        elif not (allowed & cpus):
            info["note"] = "the process's cpuset has no CPU on the GPU's node; left as is"
        else:
            info["note"] = "already confined to the GPU's node"
    except Exception as e:      # /sys not mounted, nvidia-smi missing, ...
        info["note"] = f"not bound: {type(e).__name__}: {e}"
    return info


def numa_nodes():
    """{node: set of CPUs} from sysfs ({} where it is not mounted)."""
    out = {}
    base = "/sys/devices/system/node"
    try:
        for d in os.listdir(base):
            if d.startswith("node") and d[4:].isdigit():
                cpus = set()
                for part in open(f"{base}/{d}/cpulist").read().strip().split(","):
                    if part:
                        lo, _, hi = part.partition("-")
                        cpus.update(range(int(lo), int(hi or lo) + 1))
                out[int(d[4:])] = cpus
    except OSError:
        pass
    return out


def make_matcher(ctx, res, map_xy, overlap=0):
    import gtsam_ndt_b200 as g
    m = g.NdtMatcher2D(res, device=ctx.local, stream=ctx.stream.cuda_stream, overlap=overlap)
    m.set_grid(-100.0, -100.0, 200.0, 200.0)
    t0 = time.perf_counter()
    m.set_target(map_xy)
    return m, (time.perf_counter() - t0) * 1e3


def h2d_bandwidth(ctx, h_tensor, reps=3):
    """Plain pinned-host -> device copies of the step's input, every rank at the same time: GB/s per rank."""
    torch = ctx.torch
    d = torch.empty_like(h_tensor, device=ctx.dev)
    d.copy_(h_tensor, non_blocking=True)
    ctx.sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ctx.stream)
    for _ in range(reps):
        d.copy_(h_tensor, non_blocking=True)
    e1.record(ctx.stream)
    ctx.sync_all()
    gbs = h_tensor.numel() * h_tensor.element_size() * reps / (e0.elapsed_time(e1) / 1e3) / 1e9
    return ctx.gather_floats(gbs)


def plan_upload_relay(ctx, m, gbs, min_ratio=1.15):
    """Upload relay between the ranks of the job (ndt2d_set_upload_relay): with every rank copying its step input at the same
    time, the box's host side does not feed all PCIe links alike (gbs = measured GB/s per rank). The slowest rank is paired
    with the fastest, the second slowest with the second fastest, ...; a pair whose rates differ by more than min_ratio moves
    the share x = (fast - slow) / (fast + slow) of the slow rank's chunks onto the fast rank's link (both links then finish
    together) and from that GPU over NVLink. Single node: a rank's device index is its rank. Returns the plan (same on
    every rank) or None."""
    from gtsam_ndt_b200 import distributed as D
    if ctx.world < 2 or not gbs or len(gbs) != ctx.world:
        return None
    pairs = D.upload_relay_pairs(gbs, min_ratio)
    if not pairs:
        return None
    ok = 1.0
    if ctx.rank in pairs:
        fast, x = pairs[ctx.rank]
        try:
            m.set_upload_relay(fast, min(max(x, 0.05), 0.6))
        except Exception as e:                      # e.g. no peer access on this box: every rank then stays on its own link
            print(f"[bench] rank {ctx.rank}: upload relay unavailable: {e}", file=sys.stderr)
            ok = 0.0
    if min(ctx.gather_floats(ok)) < 1.0:
        if ctx.rank in pairs:
            try:
                m.set_upload_relay(-1)
            except Exception:
                pass
        return None
    return {"pairs": {str(k): {"via_rank": v[0], "fraction": round(v[1], 3)} for k, v in pairs.items()},
            "note": "share of a slow rank's input chunks copied host -> the paired rank's GPU (its PCIe link) -> NVLink peer copy"}


def refine_upload_relay(ctx, m, plan, t_ms):
    """One calibration step: t_ms = every rank's e2e step time with the planned relay. A slow rank's time scales with the
    share 1 - x it still copies itself, its partner's with 1 + x; move x to where the two meet."""
    from gtsam_ndt_b200 import distributed as D
    for slow, v in plan["pairs"].items():
        fast, x = v["via_rank"], v["fraction"]
        ts, tf = t_ms[int(slow)], t_ms[fast]
        x2 = D.refine_relay_fraction(x, ts, tf)
        v["first_fraction"], v["fraction"] = x, round(x2, 3)
        if ctx.rank == int(slow):
            try:
                m.set_upload_relay(fast, x2)
            except Exception as e:
                print(f"[bench] rank {ctx.rank}: upload relay refinement failed, keeping {x}: {e}", file=sys.stderr)
                m.set_upload_relay(fast, x)
    plan["note"] += "; fractions refined once from the per-rank step times of a calibration run"
    return plan


def run_native(args):
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    ctx = Ctx(args)
    torch, rank, world, dev, stream = ctx.torch, ctx.rank, ctx.world, ctx.dev, ctx.stream
    K = 4 if args.overlap else 1
    sc = synth.SCAN_1080
    dense = args.world == "dense"
    if dense:
        synth.set_world(dense=True)
    ranges, poses, init, map_xy = make_workload(args, rank, dense=dense)
    xy, offsets = to_points(ranges)
    B, npts = args.scans, 1080
    m, build_ms = make_matcher(ctx, args.res, map_xy, args.overlap)
    valid_cells = int((m.cells(len(args.res) - 1)[..., 7] != 0).sum()) if rank == 0 else None

    # ---- `value`: device-resident inputs
    d_xy = torch.from_numpy(xy).to(dev)
    d_off = torch.from_numpy(offsets).to(dev)
    d_init = torch.from_numpy(np.ascontiguousarray(init)).to(dev)
    d_res = torch.zeros(B * 144, dtype=torch.uint8, device=dev)

    def step_device():
        m.align_batch_device(d_xy, d_off, B, npts, d_init, d_res)

    for _ in range(args.warmup):
        step_device()
    ctx.sync_all()
    sampler = ClockSampler(ctx.local)
    if rank == 0:
        sampler.start()
    l0 = m.kernel_launches
    ms = ctx.timed(step_device, args.steps, 0)
    launches = m.kernel_launches - l0
    res = np.frombuffer(d_res.cpu().numpy().tobytes(), dtype=g.RESULT_DTYPE)
    iters = res["iterations"].astype(np.int64)

    # ---- e2e: host buffers through the public C-ABI call, pinned memory (allocated after the NUMA binding), copies inside
    # the timed region. The primary figure uses --input; the other formats are timed as well (e2e.by_input).
    h_init = torch.from_numpy(np.ascontiguousarray(init)).pin_memory()
    h_res = torch.zeros(B * 144, dtype=torch.uint8).pin_memory()
    res_view = h_res.numpy().view(g.RESULT_DTYPE)
    U16_SCALE = 0.004  # 4 mm quantisation, 262 m maximum range
    h2d_gbs = None

    def pin(a):
        """the step's input in pinned host memory: torch's allocator, or the library's write-combined one (--pinned wc)"""
        if args.pinned == "wc":
            w = g.pinned_array(a.shape, a.dtype, write_combined=True)
            w[...] = a
            return torch.from_numpy(w)
        return torch.from_numpy(a).pin_memory()

    def e2e_run(mode):
        nonlocal h2d_gbs
        if mode == "xy":
            h_in = pin(xy)
            h_off = torch.from_numpy(offsets).pin_memory()
            nbytes = h_in.numel() * 4 + h_off.numel() * 8 + h_init.numel() * 8
            fn = lambda: m.align_batch(h_in.numpy(), h_off.numpy(), h_init.numpy(), out=res_view)
        elif mode == "ranges_u16":
            h_in = pin(np.round(ranges / U16_SCALE).clip(1, 65535).astype(np.uint16))
            nbytes = h_in.numel() * 2 + h_init.numel() * 8
            fn = lambda: m.align_batch_ranges(h_in.numpy(), sc["angle_min"], sc["angle_inc"], h_init.numpy(), range_scale=U16_SCALE, out=res_view)
        else:
            h_in = pin(ranges)
            nbytes = h_in.numel() * 4 + h_init.numel() * 8
            fn = lambda: m.align_batch_ranges(h_in.numpy(), sc["angle_min"], sc["angle_inc"], h_init.numpy(), range_scale=1.0, out=res_view)
        if mode == args.input and h2d_gbs is None:
            h2d_gbs = h2d_bandwidth(ctx, h_in)
        for _ in range(args.warmup):
            fn()
        ctx.sync_all()
        t0 = time.perf_counter()          # the call is host-synchronous: wall clock covers copies, kernels and the result read-back
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        dt_ms = (time.perf_counter() - t0) * 1e3
        same = bool(np.array_equal(res_view["iterations"], res["iterations"])) if mode != "ranges_u16" else None
        return dt_ms, int(nbytes), same

    e2e_all = {}
    relay_plan, e2e_direct = None, None
    for mode in dict.fromkeys([args.input, "xy", "ranges_f32", "ranges_u16"]):
        e2e_all[mode] = e2e_run(mode)
        if mode == args.input and args.relay == "auto":
            # the primary format once more with the upload relay between unequal ranks, if the box has any
            relay_plan = plan_upload_relay(ctx, m, h2d_gbs, float(os.environ.get("NDT2D_BENCH_RELAY_MIN_RATIO", "1.15")))
            if relay_plan:
                e2e_direct = e2e_all[mode]
                calib = e2e_run(mode)
                relay_plan = refine_upload_relay(ctx, m, relay_plan, ctx.gather_floats(calib[0]))
                e2e_all[mode] = e2e_run(mode)
    ctx.sync_all()
    e2e_ms, in_bytes, e2e_iters_equal = e2e_all[args.input]
    clocks = sampler.stop() if rank == 0 else None
    e2e_rank_ms = ctx.gather_floats(e2e_ms)
    ms, e2e_ms = ctx.max_over_ranks(ms, e2e_ms)
    e2e_direct_ms = ctx.max_over_ranks(e2e_direct[0], 0.0)[0] if relay_plan else None
    total_evals_per_step, total_scans = ctx.sum_over_ranks(float(iters.sum()), float(B))

    line = None
    if rank == 0:
        hbm, peak_src = peaks()
        kernel_ms = ms / args.steps
        alg_bytes = float(iters.sum()) * eval_bytes(npts, K)
        achieved = alg_bytes / (kernel_ms / 1e3) / 1e9
        sm_count = torch.cuda.get_device_properties(ctx.local).multi_processor_count
        key = "k_align/%s/scans=%d/res=%s/K=%d" % (args.workload, B, "-".join(str(r) for r in args.res), K)
        gp = gather_pipe(key, kernel_ms, clocks, sm_count)
        traffic = ncu_traffic("k_align", args, B)
        line = {
            "metric": METRIC, "value": total_scans * args.steps / (ms / 1e3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64 point-to-cell geometry, f32 cell-local algebra, f64 sums and solver", "data": "synthetic",
            "config": workload_config(args, B, extra={"world": args.world, "valid_map_cells": valid_cells}),
            "e2e": {"value": total_scans * args.steps / (e2e_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(in_bytes),
                    "d2h_bytes_per_step": int(B * 144), "ms_per_step": e2e_ms / args.steps, "input": args.input,
                    "api": "ndt2d_align_batch" + ("" if args.input == "xy" else "_ranges"), "iterations_equal_device_run": e2e_iters_equal,
                    "by_input": {k: {"value": B * args.steps / (v[0] / 1e3) * world, "h2d_bytes_per_step": v[1], "note": "rank 0 timing"} for k, v in e2e_all.items()},
                    "per_rank": {"h2d_gbs_plain_copy": h2d_gbs, "e2e_ms_per_step": [t / args.steps for t in e2e_rank_ms],
                                 "effective_h2d_gbs": [in_bytes / (t / args.steps / 1e3) / 1e9 for t in e2e_rank_ms],
                                 "note": "plain copy: the step's pinned input copied by every rank at the same time, no kernel; effective: input bytes / e2e step time"},
                    "numa": ctx.numa, "pinned": args.pinned, "relay": relay_plan,
                    "without_relay": ({"value": total_scans * args.steps / (e2e_direct_ms / 1e3), "ms_per_step": e2e_direct_ms / args.steps}
                                      if relay_plan else None)},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm, "traffic": traffic,
                         "dram_frac": (traffic / (kernel_ms / 1e3) / 1e9 / hbm) if traffic else None,
                         "gather_pipe_frac": gp["frac"] if gp else None,
                         "kernel": "k_align (whole LM loop per scan, one warp per scan)", "peak_source": peak_src,
                         "convention": "frac = gather traffic: every point read and 32 B cell gather counts, bytes/eval = N*(8+32K)+92 (SURVEY 8(d)); "
                                       "cells are served by L2, so frac is NOT a utilisation. dram_frac = ncu DRAM bytes per launch / kernel time / peak "
                                       "(the real HBM utilisation); gather_pipe_frac = ncu L1TEX sectors per launch / kernel time / (SMs x clock), the "
                                       "busiest unit on the memory side; `pipes` lists it beside the issue slots and the FMA pipe (no unit is saturated: "
                                       "see DESIGN.md section 5). The ncu counters are per-configuration constants from profiles/traffic.json "
                                       "(its `commit` field names the build they were captured on); the times are measured live",
                         "evals_per_launch": float(iters.sum()), "bytes_per_eval": eval_bytes(npts, K),
                         "evals_per_s": total_evals_per_step * args.steps / (ms / 1e3), "gather_pipe": gp, "pipes": ncu_pipes(key),
                         "instruction_mix": instruction_mix(key, kernel_ms, clocks, sm_count, float(iters.sum()), npts)},
            "mean_iterations": float(iters.mean()), "status_counts": np.bincount(res["status"], minlength=4).tolist(),
            "map_build_ms": build_ms, "clocks": clocks,
        }
        lat = []
        one = np.ascontiguousarray(xy[:npts])
        for i in range(60):
            t0 = time.perf_counter()
            r1 = m.align(one, init[0])
            lat.append((time.perf_counter() - t0) * 1e6)
        line["single_align_latency_us"] = {"median": float(np.median(lat[10:])), "min": float(np.min(lat[10:])),
                                           "iterations": int(r1["iterations"]), "api": "ndt2d_align (host buffers, synchronous)"}

    # ---- extra legs (default configuration only)
    failed = False
    if "prior2" in args.legs:
        leg = leg_prior2(ctx, args, m, d_xy, d_off, poses, B, npts)
        if rank == 0:
            line["prior2"] = leg
    del d_xy, d_res
    torch.cuda.empty_cache()
    if "pyramid" in args.legs:
        leg = leg_pyramid(ctx, args, map_xy)
        if rank == 0:
            line["pyramid"] = leg
    if "odometry" in args.legs:
        leg = leg_odometry(ctx, args)
        if rank == 0:
            line["odometry"] = leg
    if "sweep" in args.legs:
        leg = leg_sweep(ctx, args, m)
        failed = failed or not leg.get("ok", True)
        if rank == 0:
            line["sweep"] = leg
    if args.dump_outputs:
        dump_records(args.dump_outputs, res, rank, world)
    if rank == 0:
        os.sched_setaffinity(0, ctx.affinity0)      # the CPU legs below use every core the process was given
        if "dense" in args.legs:
            line["dense"] = leg_dense(ctx, args)
        if "config4" in args.legs:
            line["config4"] = config4_slam_frontend()
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args, xy, offsets, init, map_xy, res, m if "precision" in args.legs else None,
                                                want_config0="config0" in args.legs)
            for k in ("precision", "config0"):
                if k in line["cpu_baseline"]:
                    line[k] = line["cpu_baseline"].pop(k)
        print(json.dumps(line), flush=True)
    ctx.close()
    if failed:
        sys.exit(3)


def leg_prior2(ctx, args, m, d_xy, d_off, poses, B, npts):
    """configs[1] again from a worse prior (SURVEY 8(d): 0.2 m / 3 deg): matches/s is evaluations/s divided by the
    iteration count, and the iteration count is a function of the prior; one easy prior alone says little."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    torch = ctx.torch
    pert = synth.uniform3(B, first=ctx.rank * B + 7777777) * np.array([0.2, 0.2, math.radians(3.0)])
    d_init = torch.from_numpy(np.ascontiguousarray(poses + pert)).to(ctx.dev)
    d_res = torch.zeros(B * 144, dtype=torch.uint8, device=ctx.dev)
    ms = ctx.timed(lambda: m.align_batch_device(d_xy, d_off, B, npts, d_init, d_res), args.steps, 2)
    res = np.frombuffer(d_res.cpu().numpy().tobytes(), dtype=g.RESULT_DTYPE)
    err = np.hypot(*(res["pose"][:, :2] - poses[:, :2]).T)
    (ms,) = ctx.max_over_ranks(ms)
    scans, evals, near = ctx.sum_over_ranks(B, float(res["iterations"].sum()), float((err < 0.05).sum()))
    return {"workload": "configs[1] with prior error 0.2 m / 3 deg (single 0.25 m level, no pyramid)", "value": scans * args.steps / (ms / 1e3), "unit": UNIT,
            "ms_per_step": ms / args.steps, "mean_iterations": evals / scans, "evals_per_s": evals * args.steps / (ms / 1e3),
            "status_counts_rank0": np.bincount(res["status"], minlength=4).tolist(), "frac_within_5cm_of_truth": near / scans,
            "note": "0.2 m is most of a 0.25 m cell: without the pyramid many scans settle in a neighbouring optimum; see the pyramid leg"}


def leg_pyramid(ctx, args, map_xy):
    """BASELINE configs[2]: multi-resolution NDT (2.0/1.0/0.5 m) batched over 10 000 scans IN TOTAL, sharded over the ranks
    (strong scaling; 1250 scans per GPU at N = 8 do not fill a B200), prior error 0.2 m / 3 deg."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth, distributed as D
    torch = ctx.torch
    sc = synth.SCAN_1080
    total = 10000
    lo, hi = D.shard_range(total, ctx.rank, ctx.world)
    n = hi - lo
    ranges, poses = synth.scans(n, traj_len=total, first=lo, step=1, **sc)
    init = poses + synth.uniform3(n, first=lo + 31337) * np.array([0.2, 0.2, math.radians(3.0)])
    xy, offsets = to_points(ranges)
    m, _ = make_matcher(ctx, [2.0, 1.0, 0.5], map_xy)
    d_xy, d_off = torch.from_numpy(xy).to(ctx.dev), torch.from_numpy(offsets).to(ctx.dev)
    d_init = torch.from_numpy(np.ascontiguousarray(init)).to(ctx.dev)
    d_res = torch.zeros(n * 144, dtype=torch.uint8, device=ctx.dev)
    # 10 000 scans are 86 MB, less than the 126 MB L2: rotate through two copies of the input so that no step finds its
    # scans in the L2 left by the previous one
    d_xy2 = d_xy.clone()
    state = {"i": 0}

    def step():
        state["i"] += 1
        m.align_batch_device(d_xy if state["i"] & 1 else d_xy2, d_off, n, 1080, d_init, d_res)

    l0 = m.kernel_launches
    ms = ctx.timed(step, args.steps, max(3, args.warmup))
    launches = (m.kernel_launches - l0) * args.steps // (args.steps + max(3, args.warmup))
    res = np.frombuffer(d_res.cpu().numpy().tobytes(), dtype=g.RESULT_DTYPE)
    err = np.hypot(*(res["pose"][:, :2] - poses[:, :2]).T)
    # e2e: LaserScan ranges from pinned host memory through ndt2d_align_batch_ranges
    h_in = torch.from_numpy(ranges).pin_memory()
    h_init = torch.from_numpy(np.ascontiguousarray(init)).pin_memory()
    h_res = torch.zeros(n * 144, dtype=torch.uint8).pin_memory()
    rv = h_res.numpy().view(g.RESULT_DTYPE)
    fn = lambda: m.align_batch_ranges(h_in.numpy(), sc["angle_min"], sc["angle_inc"], h_init.numpy(), range_scale=1.0, out=rv)
    for _ in range(3):
        fn()
    ctx.sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    same = bool(rv.tobytes() == res.tobytes())
    ms, e2e_ms = ctx.max_over_ranks(ms, e2e_ms)
    evals, conv, near = ctx.sum_over_ranks(float(res["iterations"].sum()), float((res["status"] == 0).sum()), float((err < 0.05).sum()))
    m.close()
    return {"workload": "configs[2]: 2.0/1.0/0.5 m pyramid, 10000 1080-beam scans in total over %d GPU(s), prior error 0.2 m / 3 deg" % ctx.world,
            "value": total * args.steps / (ms / 1e3), "unit": UNIT, "scaling": "strong", "ms_per_step": ms / args.steps, "scans_per_gpu": n,
            "mean_iterations": evals / total, "evals_per_s": evals * args.steps / (ms / 1e3), "converged_frac": conv / total,
            "frac_within_5cm_of_truth": near / total, "gpu_launches": int(launches),
            "l2": "steps alternate between two copies of the scans (2 x %.0f MB)" % (xy.nbytes / 1e6),
            "e2e": {"value": total * args.steps / (e2e_ms / 1e3), "unit": UNIT, "ms_per_step": e2e_ms / args.steps, "h2d_bytes_per_step": int(ranges.nbytes + init.nbytes),
                    "d2h_bytes_per_step": int(n * 144), "api": "ndt2d_align_batch_ranges", "equals_device_run": same}}


def leg_odometry(ctx, args):
    """Batched scan-to-scan (ndt2d_align_pairs, the fused shared-memory path): 16 384 consecutive 1080-beam scans per GPU, 0.1 m
    apart, pair k = (scan k-1 as target, scan k as source), 0.5 m cells (configs[0]'s align, batched), prior error 2 cm / 0.2 deg."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    torch = ctx.torch
    sc = synth.SCAN_1080
    n = 16384
    ranges, poses = synth.scans(n, traj_len=3770, first=ctx.rank * 911, step=1, **sc)
    xy, offsets = to_points(ranges)
    pairs = np.stack([np.arange(n - 1), np.arange(1, n)], 1).astype(np.int32)
    c, s_ = np.cos(poses[:-1, 2]), np.sin(poses[:-1, 2])
    d = poses[1:] - poses[:-1]
    rel = np.stack([c * d[:, 0] + s_ * d[:, 1], -s_ * d[:, 0] + c * d[:, 1], d[:, 2]], 1)
    init = rel + synth.uniform3(n - 1, first=ctx.rank * n + 99) * np.array([0.02, 0.02, math.radians(0.2)])
    m = g.NdtMatcher2D([0.5], device=ctx.local, stream=ctx.stream.cuda_stream)
    d_xy, d_off = torch.from_numpy(xy).to(ctx.dev), torch.from_numpy(offsets).to(ctx.dev)
    d_init = torch.from_numpy(np.ascontiguousarray(init)).to(ctx.dev)
    d_res = torch.zeros((n - 1) * 144, dtype=torch.uint8, device=ctx.dev)
    l0 = m.kernel_launches
    ms = ctx.timed(lambda: m.align_pairs_device(d_xy, d_off, offsets, pairs, d_init, d_res), args.steps, 3)
    launches = (m.kernel_launches - l0) * args.steps // (args.steps + 3)
    res = np.frombuffer(d_res.cpu().numpy().tobytes(), dtype=g.RESULT_DTYPE)
    # the same pairs one at a time through set_target + align (what a front end without the batched call does): must be identical
    scans_list = xy.reshape(n, -1, 2)
    same = True
    for p in range(0, 64):
        m.set_target(scans_list[pairs[p, 0]])
        same = same and m.align(scans_list[pairs[p, 1]], init[p]).tobytes() == res[p].tobytes()
    (ms,) = ctx.max_over_ranks(ms)
    npairs, evals, conv, agree = ctx.sum_over_ranks(n - 1, float(res["iterations"].sum()), float((res["status"] == 0).sum()), 1.0 if same else 0.0)
    err = np.abs(res["pose"] - rel)
    m.close()
    return {"workload": "batched scan-to-scan odometry: %d consecutive 1080-beam scans per GPU, pair k = (scan k-1 -> scan k), 0.5 m cells (K=1), prior error 0.02 m / 0.2 deg" % n,
            "value": npairs * args.steps / (ms / 1e3), "unit": UNIT, "scaling": "weak", "ms_per_step": ms / args.steps, "mean_iterations": evals / npairs,
            "converged_frac": conv / npairs, "median_abs_err_vs_truth_m": float(np.median(err[:, :2])), "gpu_launches": int(launches),
            "first_64_pairs_equal_set_target_plus_align": bool(agree == ctx.world),
            "l2": "per-step scan input %.0f MB > 126 MB L2; every target's grid lives in the building warp's shared memory" % (xy.nbytes / 1e6),
            "kernel": "k_pairs_fused (one warp per pair: radix-sorted cell build in shared memory + LM loop)"}


def sweep_lattice(hyps, centre):
    """SURVEY 8(d): regular lattice, 0.2 m in x and y, 3 deg in theta, truncated to `hyps`"""
    nth = 120
    side = int(math.ceil(math.sqrt(hyps / nth)))
    gx = (np.arange(side) - side // 2) * 0.2
    lat = np.stack(np.meshgrid(gx, gx, np.radians(np.arange(nth) * 3.0 - 180.0), indexing="ij"), -1).reshape(-1, 3)[:hyps]
    return (centre + lat).astype(np.float32)


def leg_sweep(ctx, args, m):
    """BASELINE configs[3]: relocalisation, `--hyps` pose hypotheses x one 1080-pt scan vs the global map, hypotheses sharded
    over the ranks (strong scaling). Two combines of the per-rank bests are timed: peer-memory stores from the arg-max
    kernel (ndt2d_sweep_publish) and an NCCL all-gather on a side stream. Then 48 sharded queries with exact cross-shard
    ties are checked on every rank against the unsharded sweep of that rank's own GPU, and the multi-GPU relocalisation
    (sharded sweep -> global top-k -> refinement) is timed and compared with the single-GPU call."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth, distributed as D
    torch, dist, rank, world, dev, stream = ctx.torch, ctx.dist, ctx.rank, ctx.world, ctx.dev, ctx.stream
    sc = synth.SCAN_1080
    ranges, poses = synth.scans(1, traj_len=1000, first=137, **sc)
    xy = synth.polar_to_points(ranges[0], sc["angle_min"], sc["angle_inc"])
    hyp = sweep_lattice(args.hyps, poses[0])
    lo, hi = D.shard_range(len(hyp), rank, world)
    d_xy = torch.from_numpy(xy).to(dev)
    # as a leg of the default run, at least 50 queries (a step is 0.3-2 ms); as the workload, exactly --steps
    steps, warm = args.steps if args.workload == "sweep" else max(50, args.steps), max(5, args.warmup)
    # timing rule: a shard's hypotheses (12 B each) and scores (8 B) are far smaller than the 126 MB L2, so the steps
    # rotate through copies totalling more than the L2
    nrot = max(2, int(math.ceil(160e6 / max(1, (hi - lo) * 20))))
    d_hyps = [torch.from_numpy(hyp[lo:hi].copy()).to(dev) for _ in range(nrot)]
    d_scores = [torch.zeros(hi - lo, dtype=torch.float64, device=dev) for _ in range(nrot)]
    out = {"workload": "configs[3]: %d pose hypotheses (0.2 m x 0.2 m x 3 deg lattice) x one %d-pt scan vs the 200x200 m map at %s m cells, sharded over %d GPU(s)"
                       % (len(hyp), len(xy), args.res[0], world),
           "unit": "hypotheses/s", "scaling": "strong", "steps": steps, "hyps_per_gpu": hi - lo,
           "l2": "steps rotate through %d copies of the shard's hypotheses and score buffers (%.0f MB)" % (nrot, nrot * (hi - lo) * 20 / 1e6)}

    # ---- (1) peer-memory combine
    LAG, NSLOTS = 8, 64
    try:
        ex = D.PeerExchange(m, nslots=NSLOTS)
    except Exception as e:      # CUDA IPC not permitted on this box: say so, the leg fails (rc 3) but the headline line is printed
        print(f"[bench] rank {rank}: peer-memory exchange unavailable: {e}", file=sys.stderr, flush=True)
        out.update({"ok": False, "error": f"peer-memory exchange unavailable: {e}"})
        return out
    st = {"i": 0, "waited": 0, "best": None}

    def step_p2p():
        i = st["i"]
        st["i"] += 1
        ex.publish(d_xy, len(xy), d_hyps[i % nrot], hi - lo, d_scores[i % nrot], lo, i)
        if i >= LAG:
            st["best"] = ex.wait(i - LAG)
            st["waited"] = i - LAG + 1

    def drain_p2p():
        for q in range(st["waited"], st["i"]):
            st["best"] = ex.wait(q)
        st["waited"] = st["i"]

    l0 = m.kernel_launches
    ms_p2p = ctx.timed(step_p2p, steps, warm, drain_p2p)
    launches = (m.kernel_launches - l0) * steps // (steps + warm)
    _, ri, rs = m.sweep(xy, hyp, k=1, want_scores=False)           # the unsharded sweep on this rank's GPU
    same = int(st["best"][0]) == int(ri[0]) and float(st["best"][1]) == float(rs[0])
    (ms_p2p,) = ctx.max_over_ranks(ms_p2p)
    (agree,) = ctx.sum_over_ranks(1.0 if same else 0.0)
    out.update({"value": len(hyp) * steps / (ms_p2p / 1e3), "ms_per_query": ms_p2p / steps, "gpu_launches": int(launches),
                "combine": "p2p: NVLink peer stores of {index, score, epoch} from the arg-max kernel into every rank's table (ndt2d_sweep_publish); host poll %d queries behind" % LAG,
                "combine_equals_host_api_result": bool(agree == world),
                "best_hypothesis_abs_err_vs_truth": float(np.abs(hyp[int(st["best"][0])] - poses[0]).max())})

    # ---- (2) the same with an NCCL all-gather of one 16 B pair per rank on a side stream, overlapping the next sweep
    if world > 1:
        pair = [torch.zeros(2, dtype=torch.int64, device=dev) for _ in range(2)]
        gathered = [torch.zeros(2 * world, dtype=torch.int64, device=dev) for _ in range(2)]
        comm = torch.cuda.Stream(device=dev)
        ready = [torch.cuda.Event() for _ in range(2)]
        consumed = [torch.cuda.Event() for _ in range(2)]
        sn = {"i": 0, "pending": [False, False]}

        def step_nccl():
            i = sn["i"]
            sn["i"] += 1
            b = i & 1
            if sn["pending"][b]:
                stream.wait_event(consumed[b])        # the combine of query i-2 has read pair[b]
            m.sweep_device(d_xy, len(xy), d_hyps[i % nrot], hi - lo, d_scores[i % nrot], 1, pair[b].data_ptr(), pair[b].data_ptr() + 8)
            ready[b].record(stream)
            with torch.cuda.stream(comm):
                comm.wait_event(ready[b])
                dist.all_gather_into_tensor(gathered[b], pair[b])
                consumed[b].record(comm)
            sn["pending"][b] = True

        def drain_nccl():
            for b in range(2):
                if sn["pending"][b]:
                    stream.wait_event(consumed[b])

        ms_nccl = ctx.timed(step_nccl, steps, warm, drain_nccl)
        (ms_nccl,) = ctx.max_over_ranks(ms_nccl)
        gl = gathered[(sn["i"] - 1) & 1].cpu().numpy().reshape(world, 2)
        sc_ = gl[:, 1].copy().view(np.float64)
        gi = gl[:, 0] + np.array([D.shard_range(len(hyp), r, world)[0] for r in range(world)])
        order = np.lexsort((gi, -sc_))
        out["nccl"] = {"value": len(hyp) * steps / (ms_nccl / 1e3), "ms_per_query": ms_nccl / steps,
                       "combine": "nccl: all_gather_into_tensor of one (local index, score) pair per rank on a side stream",
                       "equals_p2p_result": bool(int(gi[order[0]]) == int(st["best"][0]) and float(sc_[order[0]]) == float(st["best"][1]))}

    # ---- (3) equality check: 48 sharded queries with exact cross-shard ties against the unsharded sweep of one GPU
    gx = (np.arange(41) - 20) * 0.2
    lat = np.stack(np.meshgrid(gx, gx, np.radians(np.arange(60) * 6.0 - 180.0), indexing="ij"), -1).reshape(-1, 3)
    h0 = (poses[0] + lat).astype(np.float32)
    h0 = np.concatenate([h0, h0[:997]])          # exact ties across shards: the smaller global index must win
    qbase = 1 << 20                               # query ids continue to grow: rows are reused
    nq, bad = 48, 0
    for base in range(0, nq, 8):                  # a rank is never more than one batch ahead of the slowest rank (nslots = 64)
        batch = []
        for q in range(base, base + 8):
            h = np.roll(h0, 37 * q, axis=0)
            a, b = D.shard_range(len(h), rank, world)
            d_h = torch.from_numpy(h[a:b].copy()).to(dev)
            d_s = torch.zeros(b - a, dtype=torch.float64, device=dev)
            ex.publish(d_xy, len(xy), d_h, b - a, d_s, a, qbase + q)
            batch.append((h, d_h, d_s))
        for q in range(base, base + 8):
            bi, bs = ex.wait(qbase + q, timeout_ms=30000)
            _, ri, rs = m.sweep(xy, batch[q - base][0], k=1, want_scores=False)
            if bi != int(ri[0]) or bs != float(rs[0]):
                bad += 1
                print(f"[bench] rank {rank} query {q}: exchange ({bi}, {bs}) != single GPU ({int(ri[0])}, {float(rs[0])})", file=sys.stderr, flush=True)
    (bad_total,) = ctx.sum_over_ranks(float(bad))
    out["exchange_check"] = {"queries": nq, "hypotheses_per_query": len(h0), "ranks": world, "mismatches": int(bad_total),
                             "what": "sharded ndt2d_sweep_publish + ndt2d_exchange_wait vs the unsharded ndt2d_sweep, index and score bit for bit, on every rank"}

    # ---- (4) multi-GPU relocalisation end to end: sharded sweep -> global top-k -> refinement of the k candidates
    k = 8
    reloc = D.relocalize_sharded(m, xy, hyp, k=k)           # warm-up
    ctx.sync_all()
    t0 = time.perf_counter()
    reps = 10
    for _ in range(reps):
        reloc = D.relocalize_sharded(m, xy, hyp, k=k)
    ctx.sync_all()
    reloc_ms = (time.perf_counter() - t0) * 1e3 / reps
    (reloc_ms,) = ctx.max_over_ranks(reloc_ms)
    bi1, res1 = m.relocalize(xy, hyp, k=k)                   # the single-GPU call on this rank's GPU
    same = bool(np.array_equal(reloc[0], bi1) and reloc[1].tobytes() == res1.tobytes())
    # the same through peer memory: every rank refines its own k best and stores the candidates into every rank's table;
    # one exchange per query, no collective, hypotheses resident on the device (ndt2d_relocalize_publish / _wait)
    pr = D.PeerRelocalizer(m, nslots=16, kmax=k)
    qn = {"q": 0}

    def reloc_peer():
        pr.publish(d_xy, len(xy), d_hyps[0], hi - lo, lo, k, qn["q"])
        r = pr.wait(qn["q"], k)
        qn["q"] += 1
        return r

    peer = reloc_peer()
    ctx.sync_all()
    t0 = time.perf_counter()
    for _ in range(reps):
        peer = reloc_peer()
    peer_ms = (time.perf_counter() - t0) * 1e3 / reps
    ctx.sync_all()
    pr.close()
    (peer_ms,) = ctx.max_over_ranks(peer_ms)
    same_peer = bool(np.array_equal(peer[0], bi1) and peer[1].tobytes() == res1.tobytes())
    agree, agree_peer = ctx.sum_over_ranks(1.0 if same else 0.0, 1.0 if same_peer else 0.0)
    best = reloc[1][np.lexsort((np.arange(k), -reloc[1]["score"]))[0]]
    out["relocalize"] = {"ms_per_query": peer_ms, "k": k,
                         "api": "ndt2d_relocalize_publish + ndt2d_relocalize_wait: shard sweep, its top-k and their refinement queued on the device, candidates stored into every rank's table over NVLink, local merge",
                         "equals_single_gpu_relocalize": bool(agree_peer == world),
                         "host_combine": {"ms_per_query": reloc_ms, "api": "distributed.relocalize_sharded: ndt2d_sweep from host hypotheses + torch.distributed all-gather of the top-k + ndt2d_align_batch of a share of the candidates + all-gather of the records",
                                          "equals_single_gpu_relocalize": bool(agree == world)},
                         "best_pose_abs_err_vs_truth": [float(v) for v in np.abs(best["pose"] - poses[0])]}
    out["ok"] = bool(out["combine_equals_host_api_result"] and bad_total == 0 and out["relocalize"]["equals_single_gpu_relocalize"]
                     and out["relocalize"]["host_combine"]["equals_single_gpu_relocalize"]
                     and out.get("nccl", {}).get("equals_p2p_result", True))
    ex.close()
    return out


def leg_dense(ctx, args):
    """configs[1] in the cluttered world (rank 0, one GPU): 28 k small boxes, the map holds every box edge (3.7 M points,
    > 300 k valid 0.25 m cells of 640 k), scans see ~3 m far. Fewer points share a cell and the records a batch touches no
    longer fit a few hundred KB: this is the L2-residency and sectors-per-request picture the sparse room cannot show."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    torch = ctx.torch
    sc = synth.SCAN_1080
    B = 16384
    synth.set_world(dense=True)
    try:
        map_xy = synth.dense_map()
        ranges, poses = synth.scans(B, traj_len=B, first=0, step=1, nboxes=synth.DENSE_NBOXES, **sc)
    finally:
        synth.set_world(dense=False)
    init = poses + synth.uniform3(B, first=424242) * np.array([args.perturb[0], args.perturb[0], math.radians(args.perturb[1])])
    xy, offsets = to_points(ranges)
    m, build_ms = make_matcher(ctx, args.res, map_xy)
    valid = int((m.cells(0)[..., 7] != 0).sum())
    d_xy, d_off = torch.from_numpy(xy).to(ctx.dev), torch.from_numpy(offsets).to(ctx.dev)
    d_init = torch.from_numpy(np.ascontiguousarray(init)).to(ctx.dev)
    d_res = torch.zeros(B * 144, dtype=torch.uint8, device=ctx.dev)
    fn = lambda: m.align_batch_device(d_xy, d_off, B, 1080, d_init, d_res)
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ctx.stream)
    for _ in range(args.steps):
        fn()
    e1.record(ctx.stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    res = np.frombuffer(d_res.cpu().numpy().tobytes(), dtype=g.RESULT_DTYPE)
    err = np.hypot(*(res["pose"][:, :2] - poses[:, :2]).T)
    it = float(res["iterations"].sum())
    # distinct records per 32-beam gather request at the true poses (what sets the L1TEX sector count)
    idx = m.cell_index(xy[:1080], poses[0])
    per_req = float(np.mean([len(np.unique(idx[i:i + 32])) for i in range(0, 1056, 32)]))
    m.close()
    tab = {}
    try:
        tab = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("k_align/dense/scans=%d/res=0.25/K=1" % B, {})
    except Exception:
        pass
    return {"workload": "configs[1] in the dense world: %d scans x 1080 beams vs a map with %d valid cells of 640000 (%d map points), 0.25 m, K=1, one GPU" % (B, valid, len(map_xy)),
            "value": B / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "mean_iterations": it / B, "evals_per_s": it / (ms / 1e3),
            "status_counts": np.bincount(res["status"], minlength=4).tolist(), "median_err_vs_truth_m": float(np.median(err)),
            "distinct_cells_per_32_beam_request": per_req, "map_build_ms": build_ms,
            "l2": "per-step scan input %.0f MB > 126 MB L2" % (xy.nbytes / 1e6),
            "ncu": {k: tab.get(k) for k in ("l2_hit_pct", "dram_bytes", "l1tex_sectors", "commit")} if tab else None}


def run_build(args):
    """north_star stage (1), the cell-grid build: `--map-scans` x 1080 map points binned into the 200 x 200 m lattice
    (integer accumulation with warp-level segmented reduction, then per-cell finalisation). One step = one
    ndt2d_set_target_device on device-resident points; single GPU (every rank builds its own replica of the map)."""
    import torch
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    if int(os.environ.get("RANK", "0")) != 0:
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the NDT path has no CPU fallback")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    K = 4 if args.overlap else 1
    sc = synth.SCAN_1080
    map_xy = synth.make_map(args.map_scans, traj_len=args.map_scans, **sc)
    stream = torch.cuda.current_stream()
    m = g.NdtMatcher2D(args.res, device=local, stream=stream.cuda_stream, overlap=args.overlap)
    m.set_grid(-100.0, -100.0, 200.0, 200.0)
    # rotate through copies of the point cloud totalling more than the 126 MB L2 (timing rule: inputs not L2-resident)
    nrot = max(2, int(math.ceil(160e6 / (map_xy.nbytes))))
    d_maps = [torch.from_numpy(map_xy).to(dev) for _ in range(nrot)]
    for i in range(args.warmup):
        m.set_target_device(d_maps[i % nrot], len(map_xy))
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = m.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for i in range(args.steps):
        m.set_target_device(d_maps[i % nrot], len(map_xy))
    ev1.record(stream)
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / args.steps
    launches = m.kernel_launches - l0
    # incremental update (SURVEY 8(f)-3): one scan's 1080 points added to the finished map, device-resident
    d_scan = d_maps[0][:1080].contiguous()
    for _ in range(5):
        m.add_target_device(d_scan, 1080)
    torch.cuda.synchronize()
    ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ea.record(stream)
    for _ in range(50):
        m.add_target_device(d_scan, 1080)
    eb.record(stream)
    torch.cuda.synchronize()
    add_us = ea.elapsed_time(eb) * 1e3 / 50
    # e2e: host points through ndt2d_set_target (pinned memory, copy in the timed region, host-synchronous)
    h_map = torch.from_numpy(map_xy).pin_memory()
    m.set_target(h_map.numpy())
    t0 = time.perf_counter()
    for _ in range(args.steps):
        m.set_target(h_map.numpy())
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    clocks = sampler.stop()
    ncells = sum(m.geometry(lv)["njx"] * m.geometry(lv)["njy"] for lv in range(len(args.res)))
    valid = int((m.cells(len(args.res) - 1)[..., 7] != 0).sum())
    # algorithmic bytes of one build: every point read once per level; every cell's count and five sums cleared, then
    # read and written once by the atomics' read-modify-write at least, read by the finalisation; every record written
    per_build = len(args.res) * len(map_xy) * 8 + ncells * (44 + 2 * 44 + 44 + 32)
    hbm, peak_src = peaks()
    achieved = per_build / (ms / 1e3) / 1e9
    line = {"metric": "NDT map points binned/sec (cell-grid build)", "value": len(map_xy) / (ms / 1e3), "unit": "points/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "i64 fixed-point sums, f64 finalisation, f32 records", "data": "synthetic",
            "config": {"workload": "north_star stage 1: cell-grid build, %d map points into the 200x200 m lattice at %s m cells (K=%d): %d cells, %d valid on the finest level"
                                   % (len(map_xy), "/".join(str(r) for r in args.res), K, ncells, valid),
                       "l2": "steps rotate through %d copies of the point cloud (%.0f MB > 126 MB L2)" % (nrot, nrot * map_xy.nbytes / 1e6),
                       "parallelism": "replicas only (each rank builds its own copy of the map)"},
            "e2e": {"value": len(map_xy) / (e2e_ms / 1e3), "unit": "points/s", "h2d_bytes_per_step": int(map_xy.nbytes), "d2h_bytes_per_step": 0,
                    "ms_per_step": e2e_ms, "api": "ndt2d_set_target"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm, "traffic": None,
                         "kernel": "k_accumulate + k_finalize (+ 3 clears) per level", "peak_source": peak_src, "bytes_per_build": per_build,
                         "convention": "points 8 B per level; per cell: clear 44 B, atomic read-modify-write 88 B, finalise read 44 B, record 32 B"},
            "incremental_update_us": {"value": add_us, "what": "ndt2d_add_target_device of one 1080-point scan into the finished map (accumulate + finalise), per call"},
            "clocks": clocks}
    print(json.dumps(line), flush=True)


def run_odometry(args):
    """Batched scan-to-scan odometry (ndt2d_align_pairs): `--scans` consecutive 1080-beam scans of the trajectory, pair
    k = (scan k-1 as target, scan k as source), prior = true relative motion + `--perturb`. One step = every target's
    grid built (one warp per target and level, hash tables) + every pair aligned. BASELINE configs[0] is the single
    CPU case of this align (scan-to-scan, 0.5 m cells); the batched form is what a log or a set of loop-closure
    candidates needs. Single GPU (pairs would shard like scans)."""
    import torch
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    if int(os.environ.get("RANK", "0")) != 0:
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the NDT path has no CPU fallback")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    K = 4 if args.overlap else 1
    sc = synth.SCAN_1080
    n = args.scans
    ranges, poses = synth.scans(n, traj_len=3770, first=0, step=1, **sc)      # the 377 m loop in 0.1 m steps (laps repeat with new noise)
    xy, offsets = to_points(ranges)
    pairs = np.stack([np.arange(n - 1), np.arange(1, n)], 1).astype(np.int32)
    c, s_ = np.cos(poses[:-1, 2]), np.sin(poses[:-1, 2])
    d = poses[1:] - poses[:-1]
    rel = np.stack([c * d[:, 0] + s_ * d[:, 1], -s_ * d[:, 0] + c * d[:, 1], d[:, 2]], 1)
    init = rel + synth.uniform3(n - 1) * np.array([args.perturb[0], args.perturb[0], math.radians(args.perturb[1])])
    stream = torch.cuda.current_stream()
    m = g.NdtMatcher2D(args.res, device=local, stream=stream.cuda_stream, overlap=args.overlap)
    d_xy = torch.from_numpy(xy).to(dev)
    d_off = torch.from_numpy(offsets).to(dev)
    d_init = torch.from_numpy(np.ascontiguousarray(init)).to(dev)
    d_res = torch.zeros((n - 1) * 144, dtype=torch.uint8, device=dev)
    for _ in range(args.warmup):
        m.align_pairs_device(d_xy, d_off, offsets, pairs, d_init, d_res)
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = m.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        m.align_pairs_device(d_xy, d_off, offsets, pairs, d_init, d_res)
    ev1.record(stream)
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / args.steps
    launches = m.kernel_launches - l0
    res = np.frombuffer(d_res.cpu().numpy().tobytes(), dtype=g.RESULT_DTYPE)
    # e2e: pinned host scans through ndt2d_align_pairs, copies and result read-back in the timed region
    h_xy = torch.from_numpy(xy).pin_memory()
    m.align_pairs(h_xy.numpy(), offsets, pairs, init)
    t0 = time.perf_counter()
    reps = max(1, args.steps // 2)
    for _ in range(reps):
        rh = m.align_pairs(h_xy.numpy(), offsets, pairs, init)
    e2e_ms = (time.perf_counter() - t0) * 1e3 / reps
    clocks = sampler.stop()
    # the same pairs one at a time through set_target + align (what a front end without the batched call does)
    t0 = time.perf_counter()
    nseq = min(256, n - 1)
    scans_list = xy.reshape(n, -1, 2)
    same = True
    for p in range(nseq):
        m.set_target(scans_list[pairs[p, 0]])
        one = m.align(scans_list[pairs[p, 1]], init[p])
        same = same and one.tobytes() == res[p].tobytes()
    seq_ms = (time.perf_counter() - t0) * 1e3 / nseq
    err = res["pose"] - rel
    good = res["status"] == 0
    iters = res["iterations"].astype(np.int64)
    hbm, peak_src = peaks()
    alg_bytes = float(iters.sum()) * eval_bytes(1080, K)
    achieved = alg_bytes / (ms / 1e3) / 1e9
    line = {"metric": "NDT scan-to-scan matches/sec (1080-pt 2D scans, batched pairs)", "value": (n - 1) / (ms / 1e3), "unit": "matches/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 per point, f64 sums and solver", "data": "synthetic",
            "config": {"workload": "batched scan-to-scan odometry: %d consecutive 1080-beam scans 0.1 m apart, pair k = (scan k-1 -> scan k), %s m cells (K=%d), "
                                   "per-target grids in hash tables, prior error %.2f m / %.1f deg" % (n, "/".join(str(r) for r in args.res), K, args.perturb[0], args.perturb[1]),
                       "l2": "per-step scan input %.0f MB; per-target tables %.1f GB are rebuilt every step" % (xy.nbytes / 1e6, (n - 1) * len(args.res) * 4097 * 76 / 1e9),
                       "parallelism": "replicas only in this bench (pairs shard like scans)"},
            "e2e": {"value": (n - 1) / (e2e_ms / 1e3), "unit": "matches/s", "h2d_bytes_per_step": int(xy.nbytes + offsets.nbytes + init.nbytes),
                    "d2h_bytes_per_step": int((n - 1) * 144), "ms_per_step": e2e_ms, "api": "ndt2d_align_pairs",
                    "equals_device_run": bool(rh.tobytes() == res.tobytes())},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm, "traffic": None,
                         "kernel": "k_align<PAIRS> (hash-table gathers) after k_pairs_build", "peak_source": peak_src,
                         "bytes_per_eval": eval_bytes(1080, K), "evals_per_launch": float(iters.sum()),
                         "convention": "gather traffic (DESIGN.md section 4); the build's traffic is not counted"},
            "mean_iterations": float(iters.mean()), "status_counts": np.bincount(res["status"], minlength=4).tolist(),
            "median_abs_err_vs_truth_m": float(np.median(np.abs(err[good, :2]))) if good.any() else None,
            "sequential_set_target_plus_align": {"ms_per_pair": seq_ms, "pairs": nseq, "bit_identical_to_batched": bool(same)},
            "clocks": clocks}
    print(json.dumps(line), flush=True)


def run_newton(args):
    """north_star stage (2) in isolation: the Newton-step evaluation (score, 3-gradient, 3x3 Hessian) of one 1080-point
    scan at `--hyps` poses scattered like LM iterates around the true pose (k_eval_poses<FULL>, ndt2d_evaluate_device).
    This is SURVEY.md 8(d)'s unit of work with no solver and no iteration control around it. Single GPU."""
    import torch
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    if int(os.environ.get("RANK", "0")) != 0:
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the NDT path has no CPU fallback")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    K = 4 if args.overlap else 1
    sc = synth.SCAN_1080
    map_xy = synth.make_map(args.map_scans, traj_len=args.map_scans, **sc)
    ranges, poses = synth.scans(1, traj_len=1000, first=137, **sc)
    xy = synth.polar_to_points(ranges[0], sc["angle_min"], sc["angle_inc"])
    npose = args.hyps
    rng = np.random.default_rng(7)
    P = poses[0] + rng.normal(size=(npose, 3)) * np.array([0.03, 0.03, math.radians(0.3)])
    stream = torch.cuda.current_stream()
    m = g.NdtMatcher2D(args.res, device=local, stream=stream.cuda_stream, overlap=args.overlap)
    m.set_grid(-100.0, -100.0, 200.0, 200.0)
    m.set_target(map_xy)
    d_xy = torch.from_numpy(xy).to(dev)
    nrot = max(2, int(math.ceil(160e6 / (npose * (24 + 80 + 4)))))      # poses in, sums and counts out: rotate beyond the L2
    d_P = [torch.from_numpy(P).to(dev) for _ in range(nrot)]
    d_out = [torch.zeros(npose * 10, dtype=torch.float64, device=dev) for _ in range(nrot)]
    d_cnt = [torch.zeros(npose, dtype=torch.int32, device=dev) for _ in range(nrot)]
    for i in range(args.warmup):
        m.evaluate_device(d_xy, len(xy), d_P[i % nrot], npose, d_out[i % nrot], d_cnt[i % nrot])
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = m.kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for i in range(args.steps):
        m.evaluate_device(d_xy, len(xy), d_P[i % nrot], npose, d_out[i % nrot], d_cnt[i % nrot])
    ev1.record(stream)
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / args.steps
    launches = m.kernel_launches - l0
    # e2e: host poses in, host sums out, through ndt2d_evaluate (pinned memory, copies in the timed region)
    h_P = torch.from_numpy(P).pin_memory()
    m.evaluate(xy, h_P.numpy())
    t0 = time.perf_counter()
    for _ in range(max(1, args.steps // 5)):
        out, cnt = m.evaluate(xy, h_P.numpy())
    e2e_ms = (time.perf_counter() - t0) * 1e3 / max(1, args.steps // 5)
    clocks = sampler.stop()
    dev_out = d_out[(args.steps - 1) % nrot].cpu().numpy().reshape(npose, 10)
    per_eval = eval_bytes(len(xy), K)
    hbm, peak_src = peaks()
    achieved = npose * per_eval / (ms / 1e3) / 1e9
    line = {"metric": "NDT Newton-step evaluations/sec (1080-pt scan: score, gradient, Hessian)", "value": npose / (ms / 1e3), "unit": "evaluations/s",
            "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 per point, f64 sums", "data": "synthetic",
            "config": {"workload": "north_star stage 2: Newton-step kernel alone, one %d-pt scan at %d poses (sigma 3 cm / 0.3 deg around the truth) vs 200x200 m map at %s m cells (K=%d)"
                                   % (len(xy), npose, args.res[0], K),
                       "l2": "steps rotate through %d copies of the pose and result buffers (%.0f MB > 126 MB L2); the scan and the cell table are cache-resident by design"
                             % (nrot, nrot * npose * 108 / 1e6),
                       "parallelism": "replicas only"},
            "e2e": {"value": npose / (e2e_ms / 1e3), "unit": "evaluations/s", "h2d_bytes_per_step": int(npose * 24 + len(xy) * 8),
                    "d2h_bytes_per_step": int(npose * 84), "ms_per_step": e2e_ms, "api": "ndt2d_evaluate",
                    "equals_device_run": bool(np.array_equal(out, dev_out))},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm, "traffic": None,
                         "kernel": "k_eval_poses<FULL> (one warp per pose, scan staged per block)", "peak_source": peak_src, "bytes_per_eval": per_eval,
                         "convention": "gather traffic (DESIGN.md section 4): every point read and 32 B record gather counts; scan and cells are cache-resident"},
            "clocks": clocks}
    print(json.dumps(line), flush=True)


def run_sweep(args):
    """`--workload sweep`: the sweep leg on its own, as one bench line (metric: pose hypotheses/s)."""
    from gtsam_ndt_b200 import synth
    ctx = Ctx(args)
    sc = synth.SCAN_1080
    map_xy = synth.make_map(args.map_scans, traj_len=args.map_scans, **sc)
    m, _ = make_matcher(ctx, args.res, map_xy, args.overlap)
    sampler = ClockSampler(ctx.local)
    if ctx.rank == 0:
        sampler.start()
    leg = leg_sweep(ctx, args, m)
    clocks = sampler.stop() if ctx.rank == 0 else None
    if ctx.rank == 0:
        K = 4 if args.overlap else 1
        hbm, peak_src = peaks()
        per_hyp = 1080 * (8 + 32 * K) + 12 + 8
        achieved = leg["hyps_per_gpu"] * per_hyp / (leg["ms_per_query"] / 1e3) / 1e9
        key = "k_eval_poses/sweep/hyps=%d/res=%s/K=%d" % (args.hyps, "-".join(str(r) for r in args.res), K)
        sm_count = ctx.torch.cuda.get_device_properties(ctx.local).multi_processor_count
        line = {"metric": "NDT pose hypotheses/sec (1080-pt scan vs global map)", "value": leg["value"], "unit": "hypotheses/s", "n_gpus": ctx.world,
                "steps": leg["steps"], "warmup": max(5, args.warmup), "ms_per_step": leg["ms_per_query"], "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64 point-to-cell geometry, f32 cell-local algebra, f64 sums", "data": "synthetic",
                "config": {"workload": leg["workload"], "l2": leg["l2"], "parallelism": "hypotheses sharded per GPU; " + leg["combine"]},
                "e2e": {"value": args.hyps / (leg["relocalize"]["ms_per_query"] / 1e3), "unit": "hypotheses/s", "h2d_bytes_per_step": int(leg["hyps_per_gpu"] * 12 + 1080 * 8),
                        "d2h_bytes_per_step": int(8 * (16 + 144)), "ms_per_step": leg["relocalize"]["ms_per_query"],
                        "api": "relocalisation from host buffers: " + leg["relocalize"]["api"]},
                "gpu_launches": leg["gpu_launches"],
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
                             "traffic": ncu_traffic_sweep(args, args.hyps) if ctx.world == 1 else None, "kernel": "k_eval_poses (score only)",
                             "peak_source": peak_src, "bytes_per_hypothesis": per_hyp,
                             "gather_pipe": gather_pipe(key, leg["ms_per_query"], clocks, sm_count) if ctx.world == 1 else None,
                             "convention": "gather traffic (see DESIGN.md section 4); scan and cells are cache-resident"},
                "sweep": leg, "clocks": clocks}
        print(json.dumps(line), flush=True)
    ctx.close()
    if not leg["ok"]:
        sys.exit(3)


def cpu_baseline(args, xy, offsets, init, map_xy, res_gpu, matcher=None, want_config0=False):
    """The CPU checkers on rank 0 (the one place besides --impl reference where bench.py executes oracle/):
    the spec oracle on a bounded sample of the same workload, all host threads (reported, not the target); with `matcher`,
    the distance of the GPU results from the independent f64 twin (`precision`); with want_config0, BASELINE configs[0]."""
    import oracle
    o = oracle.Oracle(args.res, overlap=args.overlap)
    o.set_grid(-100.0, -100.0, 200.0, 200.0)
    o.set_target(map_xy)
    cores = host_cores()
    probe = min(len(offsets) - 1, 8 * cores)
    t0 = time.perf_counter()
    o.align_batch(xy, offsets[: probe + 1], init[:probe], nthreads=cores)
    rate = probe / (time.perf_counter() - t0)
    n = args.cpu_sample or int(min(len(offsets) - 1, max(probe, rate * 12.0)))
    t0 = time.perf_counter()
    reps = 0
    while True:
        r = o.align_batch(xy, offsets[: n + 1], init[:n], nthreads=cores)
        reps += 1
        dt = time.perf_counter() - t0
        if dt >= 10.0 or reps >= 64:
            break
    dp = np.abs(r["pose"] - res_gpu["pose"][:n]).max()
    out = {"value": n * reps / dt, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": f"first {n} scans of the step x {reps} passes, CPU spec oracle (SPEC.md port), {dt:.1f} s",
           "max_abs_pose_diff_vs_gpu": float(dp), "iterations_equal": bool(np.array_equal(r["iterations"], res_gpu["iterations"][:n])),
           "records_identical": bool(r.tobytes() == res_gpu[:n].tobytes())}
    if matcher is not None:
        out["precision"] = precision_vs_f64(matcher, map_xy, xy, offsets, init)
    if want_config0:
        out["config0"] = config0_pair(matcher.device if matcher is not None else 0)
    return out


def precision_vs_f64(m, map_xy, xy, offsets, init, n=64):
    """GPU evaluate / align on configs[1] against oracle/f64ref.py (an independent f64 NDT that follows none of SPEC.md's
    bit-level choices), at north_star's tolerances: score and Hessian 1e-6 relative, pose 1e-5 m / 1e-6 rad."""
    from oracle import f64ref
    tw = f64ref.NdtF64([m.geometry(0)])
    tw.set_target(map_xy)
    sel = np.linspace(0, len(offsets) - 2, n).astype(int)
    scans = [xy[offsets[i]:offsets[i + 1]] for i in sel]
    twin = [tw.align(s, init[i]) for s, i in zip(scans, sel)]
    sr, hr, cells_equal = [], [], 0
    for s, t in zip(scans, twin):
        out, cnt = m.evaluate(s, t["pose"])
        H = np.array([[out[4], out[5], out[6]], [out[5], out[7], out[8]], [out[6], out[8], out[9]]])
        sr.append(abs(out[0] - t["score"]) / t["score"])
        hr.append(np.abs(H - t["hessian"]).max() / np.abs(t["hessian"]).max())
        cells_equal += int(cnt == t["count"])
    r = m.align_batch(np.concatenate(scans), np.concatenate([[0], np.cumsum([len(s) for s in scans])]), init[sel])
    d = r["pose"] - np.array([t["pose"] for t in twin])
    dpos = np.hypot(d[:, 0], d[:, 1])
    drot = np.abs((d[:, 2] + np.pi) % (2 * np.pi) - np.pi)
    ok = (dpos <= 1e-5) & (drot <= 1e-6)
    return {"against": "oracle/f64ref.py: independent double-precision NDT (numpy), same algorithm, none of SPEC.md's bit-level choices; parity unpinned (no reference source)",
            "scans": n, "evaluate_at_f64_optimum": {"score_rel_max": float(max(sr)), "score_rel_median": float(np.median(sr)),
                                                    "hessian_rel_max": float(max(hr)), "hessian_rel_median": float(np.median(hr)),
                                                    "same_contributing_pairs": cells_equal},
            "align_vs_f64_lm": {"within_1e-5m_1e-6rad": float(ok.mean()), "same_iteration_count": float(np.mean(r["iterations"] == np.array([t["iterations"] for t in twin]))),
                                "dpos_median": float(np.median(dpos)), "dpos_p90": float(np.percentile(dpos, 90)), "dpos_max": float(dpos.max()),
                                "drot_median": float(np.median(drot)), "drot_max": float(drot.max())},
            "tolerance": {"score_hessian_rel": 1e-6, "pose_m": 1e-5, "pose_rad": 1e-6},
            "note": "scans outside the pose tolerance took a different accept/reject path through the LM loop (DESIGN.md section 3b); SPEC v3 measured 1.3e-4 / 7e-3 on score / Hessian"}


def config4_slam_frontend():
    """BASELINE configs[4], the part that exists without GTSAM: examples/slam_frontend.cpp (C++ host code over ndt2d.hpp) drives a
    closed loop through a synthetic room - sequential GPU NDT odometry, the loop-closure search (sweep + refinement), the same
    odometry batched through alignPairs - checks its own factors against the truth and writes the g2o pose graph that
    gtsam::readG2o + ISAM2 consume. Built with the system g++ on the spot, in a temporary directory (the tree may be
    read-only); the figures are the program's own."""
    import re
    import tempfile
    src = os.path.join(ROOT, "examples", "slam_frontend.cpp")
    libdir = os.path.join(ROOT, "gtsam_ndt_b200")
    try:
        with tempfile.TemporaryDirectory() as td:
            exe = os.path.join(td, "slam_frontend")
            subprocess.run(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), src, "-L", libdir, "-lndt2d",
                            "-Wl,-rpath," + libdir, "-o", exe], check=True, capture_output=True, timeout=120)
            r = subprocess.run([exe, os.path.join(td, "graph.g2o")], capture_output=True, text=True, timeout=120)
        out = r.stdout
        num = lambda rx: [float(x) for x in re.search(rx, out).groups()]
        edges, bad, worst, drift = num(r"odometry: (\d+) edges, (\d+) not converged, worst relative error ([\d.]+) m, dead-reckoning drift ([\d.]+) m")
        odo_ms, loop_ms, nhyp = num(r"timing: ([\d.]+) ms per odometry step .*?, ([\d.]+) ms for the loop-closure search \((\d+) hypotheses")
        npairs, batch_ms, differ = num(r"batched odometry: (\d+) pairs in ([\d.]+) ms through alignPairs .*?, (\d+) results differ")
        loop_err = num(r"loop closure .*?error vs truth ([\d.]+) m")[0]
        return {"workload": "configs[4] front end: examples/slam_frontend (C++ over ndt2d.hpp), closed loop in a 24 x 16 m room, GPU odometry + "
                            "loop closure -> g2o pose graph for GTSAM (no solver here: GTSAM is absent)",
                "ok": r.returncode == 0, "odometry_edges": int(edges), "not_converged": int(bad), "worst_relative_error_m": worst,
                "dead_reckoning_drift_m": drift, "loop_closure_error_m": loop_err, "ms_per_odometry_step_sequential": odo_ms,
                "odometry_steps_per_s_sequential": 1e3 / odo_ms, "loop_closure_search_ms": loop_ms, "loop_closure_hypotheses": int(nhyp),
                "batched_odometry_ms": batch_ms, "batched_odometry_pairs_per_s": npairs / (batch_ms / 1e3),
                "batched_results_differing_from_sequential": int(differ)}
    except Exception as e:
        return {"workload": "configs[4] front end: examples/slam_frontend", "ok": False, "error": repr(e)[:300]}


def config0_pair(device=0):
    """BASELINE configs[0]: one synthetic 360-beam scan-to-scan align at 0.5 m cells; the CPU oracle on one thread next to
    the GPU's single-align latency through the host API (set_target of the previous scan + align of the new one)."""
    import oracle
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    sc = synth.SCAN_360
    ranges, poses = synth.scans(2, traj_len=3770, first=100, step=1, **sc)          # 0.1 m apart on the loop
    a, b = (synth.polar_to_points(ranges[i], sc["angle_min"], sc["angle_inc"]) for i in (0, 1))
    c, s_ = math.cos(poses[0, 2]), math.sin(poses[0, 2])
    d = poses[1] - poses[0]
    rel = np.array([c * d[0] + s_ * d[1], -s_ * d[0] + c * d[1], d[2]])
    init = rel + np.array([0.10, -0.05, math.radians(2.0)])                          # SURVEY 8(d) offset for config 1
    o = oracle.Oracle([0.5])
    t0 = time.perf_counter()
    reps = 0
    while time.perf_counter() - t0 < 1.0:
        o.set_target(a)
        ro = o.align(b, init)
        reps += 1
    cpu_ms = (time.perf_counter() - t0) * 1e3 / reps
    m = g.NdtMatcher2D([0.5], device=device)
    lat, lat_align = [], []
    for i in range(80):
        t0 = time.perf_counter()
        m.set_target(a)
        t1 = time.perf_counter()
        rg = m.align(b, init)
        t2 = time.perf_counter()
        lat.append((t2 - t0) * 1e3)
        lat_align.append((t2 - t1) * 1e3)
    m.close()
    return {"workload": "configs[0]: single 360-beam scan-to-scan NDT align, 0.5 m cells, prior error 0.10 m / -0.05 m / 2 deg",
            "cpu_oracle_1_thread_ms": cpu_ms, "gpu_set_target_plus_align_ms": float(np.median(lat[10:])), "gpu_align_only_ms": float(np.median(lat_align[10:])),
            "iterations": int(rg["iterations"]), "status": int(rg["status"]), "records_identical": bool(rg.tobytes() == ro.tobytes()),
            "err_vs_truth": [float(v) for v in np.abs(rg["pose"] - rel)],
            "note": "a single 360-point align is latency, not throughput: one block runs the LM loop; host API, synchronous, pageable buffers"}


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload == "sweep":
        run_sweep(a)
    elif a.workload == "build":
        run_build(a)
    elif a.workload == "newton":
        run_newton(a)
    elif a.workload == "odometry":
        run_odometry(a)
    else:
        run_native(a)
