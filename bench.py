#!/usr/bin/env python
"""bench.py — Mpts/s of one full MapEval metric pass (AC + CD + full CD + MME + voxel Gaussians + AWD + SCS).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C3] [--impl reference] [--dump-outputs DIR]

A step = one pass of the hot path over one synthetic cloud pair (SURVEY.md §8d): both lattices are laid out from
the fp64 clouds, NN est->gt and gt->est with the five-threshold accumulators and the full-Chamfer sums, MME of the
estimated map (and of the GT map when the config says so), per-voxel Gaussians, AWD and SCS.
  value : est points / step time with both clouds already resident in HBM (device-resident arm)
  e2e   : the same pass through the C-ABI with HOST (pinned) buffers: H2D of both clouds and D2H of the result
          structs are inside the timed region
N > 1 (torchrun, one rank per GPU): slab layout — every rank lays out and evaluates only the voxel layers it owns of both
clouds (lattice builds, sweeps and voxel stage sharded; `--layout replicated`: whole lattices on every rank, query ranges
sharded; scenes that cannot be cut fall back to it), the W table of the voxel stage is MAX-all-reduced and the
sum-reducible accumulators are all-reduced in place over NCCL once per step (strong scaling: the cloud pair is fixed).  Timing: CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.
`--impl reference` times the CPU restatement of the reference (oracle/, all host threads) on the SAME workload as the
CUDA arm (C3 by default: 10 M vs 10 M); its timed passes are capped by wall time (REF_BUDGET_S) and the line says how
many ran.  `e2e_pageable` repeats the e2e arm from plain (pageable) numpy memory, the way a std::vector caller hands
the clouds over.  For N > 1 the e2e arm uploads 1/N of each cloud per rank and all-gathers over NVLink (NCCL).
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

from cloud_map_evaluation_b200 import _abi as A  # noqa: E402
from cloud_map_evaluation_b200 import synth  # noqa: E402

METRIC = "Mpts/s full AC+CD+AWD+MME pass"
UNIT = "Mpts/s"


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _profile_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu summary, if present."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


class ClockSampler:
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sel = [r for (ts, r) in self.rows if t0 - 0.05 <= ts <= t1 + 0.15] or [r for (_, r) in self.rows]
        sm, smax, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in sel:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except Exception:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


VOXEL_HASH_NOTE = ("voxel maps keyed with a mixing hash instead of the reference's XOR hash (voxel_calculator.hpp:18-22), whose "
                   "collisions make the reference-faithful voxel stage of C3 take 444 s (tests/golden/c3_oracle.json, oracle_seconds): "
                   "this baseline is FASTER than the reference's own code; same voxel Gaussians, AWD / SCS equal to 1e-15")


def _cpu_pass(est, gt, cfg, threads, faithful=False):
    """One full pass with the oracle (the CPU restatement of the reference).  faithful=True keeps the reference's own
    threading: serial 1-NN loops on path A (map_eval.cpp:1215-1236), TBB / OpenMP for the estimated map's MME
    (:1716-1717), serial MME of the ground truth (:1451) — and its XOR voxel hash; otherwise every sweep uses all `threads`
    and the voxel maps a mixing hash (VOXEL_HASH_NOTE)."""
    from oracle import oracle as O
    p = A.make_nn_params(cfg["tau"], 1.0)
    O.set_voxel_hash(not faithful)
    t0 = time.perf_counter()
    O.eval_nn(est, gt, p, threads=1 if faithful else threads)
    if cfg["mme"]:
        O.eval_mme(est, cfg["nn_radius"], 10, threads=threads)
        if cfg["gt_mme"]:
            O.eval_mme(gt, cfg["nn_radius"], 5, threads=1 if faithful else threads)
    if cfg["awd"]:
        O.eval_awd(est, gt, cfg["vmd_voxel_size"], 100, 5)
    dt = time.perf_counter() - t0
    O.set_voxel_hash(False)
    return dt


def _host_threads():
    """All the host threads this process may use.  (Under torchrun OMP_NUM_THREADS is forced to 1 per rank, which
    omp_get_max_threads() would report; the CPU arm runs on rank 0 alone and takes the cores of the box.)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def _cpu_sample(name, target_pts=1_000_000):
    base = synth.CONFIGS[name]
    scale = min(1.0, target_pts / base["n_est"])
    est, gt, cfg = synth.make_pair(name, scale=scale)
    return est, gt, cfg, scale


REF_BUDGET_S = 150.0      # wall-time cap of the reference arm's timed passes (the driver allows minutes, not hours)


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (oracle port: Open3D/Eigen/TBB are absent, SURVEY §8c) on the same
    config as the CUDA arm, at full size.  One pass over 10 M vs 10 M points takes the better part of a minute on 128
    cores (with the voxel maps on a mixing hash — VOXEL_HASH_NOTE; 8 minutes with the reference's own hash), so the number of
    timed passes is capped by wall time; `steps` is what actually ran."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O  # noqa: F401
    threads = _host_threads()
    est, gt, cfg = synth.make_pair(args.config, scale=args.scale)
    times = []
    t_begin = time.perf_counter()
    for k in range(max(1, args.steps)):
        times.append(_cpu_pass(est, gt, cfg, threads))
        if time.perf_counter() - t_begin + times[-1] > REF_BUDGET_S:
            break
    dt = float(np.mean(times))
    v = len(est) / dt / 1e6
    # SURVEY §8d mode (1), the reference's own threading (serial 1-NN loops, serial GT MME) and voxel hash: on a 1 M-point
    # sample only — at full size the serial loops alone take minutes and the voxel-map build 7 more.
    s_est, s_gt, s_cfg, s_scale = _cpu_sample(args.config)
    dt_f = _cpu_pass(s_est, s_gt, s_cfg, threads, faithful=True)
    sample = (f"{args.config} at full size ({len(est)} est vs {len(gt)} gt points), full pass, all-cores mode, "
              f"{len(times)} timed pass(es) of {args.steps} requested (wall-time cap {REF_BUDGET_S:.0f} s), no warm-up pass")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "steps_requested": args.steps, "warmup": 0, "warmup_requested": args.warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.config}: {synth.CONFIGS[args.config]['desc']}", "n_est": len(est), "n_gt": len(gt),
                   "tau": cfg["tau"], "icp_max_distance": 1.0, "nn_radius": cfg["nn_radius"],
                   "vmd_voxel_size": cfg["vmd_voxel_size"], "mme_gt": bool(cfg["gt_mme"]), "generated": "numpy",
                   "sample": sample},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "pass_seconds": times, "voxel_hash": VOXEL_HASH_NOTE,
                         "reference_faithful_pass_seconds_c3": "485 (NN 18 + MME 23 + voxel stage 444; B200 host, 128 threads, "
                                                               "tests/golden/c3_oracle.json)",
                         "reference_threading_value": len(s_est) / dt_f / 1e6,
                         "reference_threading": f"serial 1-NN loops and GT MME as the reference runs them, est MME on all cores, XOR voxel hash; "
                                                f"{args.config} at scale {s_scale:g} ({len(s_est)} points)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def _alloc_pinned(t):
    return t.pin_memory()


def _dump_outputs(out_dir, res):
    """Writes the result structs of one pass as DIR/<struct>.<field>.npy, one float64 array per field (the integer
    counts are exact in float64).  The clouds are generated from fixed seeds, so two builds run with the same arguments
    can be compared file by file."""
    outs = {"nn": A.struct_to_dict(res["nn"]), "n_far": list(res["n_far"])}
    for m, side in zip(res["mme"], ("est", "gt")):
        outs[f"mme_{side}"] = A.struct_to_dict(m)
    if res["awd"] is not None:
        outs["awd"] = A.struct_to_dict(res["awd"])
    os.makedirs(out_dir, exist_ok=True)

    def write(name, v):
        if isinstance(v, dict):
            for k, x in v.items():
                write(f"{name}.{k}", x)
        else:
            np.save(os.path.join(out_dir, name + ".npy"), np.asarray(v, dtype=np.float64))

    for name, v in outs.items():
        write(name, v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="C3", choices=sorted(synth.CONFIGS))
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (debugging only; not a bench line)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--layout", default="slab", choices=["slab", "replicated"],
                    help="N > 1: slab = every rank lays out only the voxel layers it owns (default); replicated = whole clouds on every rank")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer arms (large configs on small hosts)")
    ap.add_argument("--gen", default="auto", choices=["auto", "numpy", "device"],
                    help="where the synthetic clouds are generated (auto: on the device above 20 M points)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the device-resident arm returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA arm only")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
        return

    # exactly ONE line may reach stdout (the JSON record): libraries that print there (NCCL's version banner) are sent
    # to stderr for the duration of the run
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    from cloud_map_evaluation_b200 import api
    from cloud_map_evaluation_b200 import dist as mdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libmapeval_b200 has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    sampler = ClockSampler(local_rank) if rank == 0 else None   # nvidia-smi needs ~1 s to start: launch it early
    base = synth.CONFIGS[args.config]
    gen = args.gen
    if gen == "auto":
        gen = "device" if max(base["n_est"], base["n_gt"]) * args.scale > 20_000_000 else "numpy"
    if gen == "device":
        from cloud_map_evaluation_b200 import synth_torch
        d_est, d_gt, cfg = synth_torch.make_pair(args.config, scale=args.scale, device=dev)
    else:
        est, gt, cfg = synth.make_pair(args.config, scale=args.scale)
        d_est = torch.from_numpy(est).to(dev)
        d_gt = torch.from_numpy(gt).to(dev)
    n_est, n_gt = d_est.shape[0], d_gt.shape[0]
    p = A.make_nn_params(cfg["tau"], 1.0)        # path A as written + full CD (SURVEY §8d)

    # host copies for the e2e arms.  N = 1: the whole clouds, pinned (e2e) and pageable (e2e_pageable).  N > 1: every
    # rank holds 1/N of each cloud on its host side, uploads that slice over its own PCIe link and the slices are
    # all-gathered over NVLink (NCCL) — the full 480 MB no longer crosses every rank's PCIe link.
    do_e2e = not args.no_e2e
    m_est, m_gt = -(-n_est // world), -(-n_gt // world)          # slice lengths (last slice padded)
    h_est = h_gt = p_est = p_gt = None
    g_est = g_gt = s_est = s_gt = None
    if do_e2e:
        def host_slice(d_full, m):
            lo, hi = rank * m, min(d_full.shape[0], (rank + 1) * m)
            h = torch.zeros((m, 3), dtype=torch.float64)
            if hi > lo:
                h[:hi - lo] = d_full[lo:hi].cpu()
            return h
        if world == 1:
            h_est, h_gt = d_est.cpu(), d_gt.cpu()
            p_est, p_gt = h_est.numpy().copy(), h_gt.numpy().copy()        # plain pageable memory
            h_est, h_gt = _alloc_pinned(h_est), _alloc_pinned(h_gt)
        else:
            h_est, h_gt = _alloc_pinned(host_slice(d_est, m_est)), _alloc_pinned(host_slice(d_gt, m_gt))
            g_est = torch.empty((world * m_est, 3), dtype=torch.float64, device=dev)
            g_gt = torch.empty((world * m_gt, 3), dtype=torch.float64, device=dev)
            s_est = torch.empty((m_est, 3), dtype=torch.float64, device=dev)      # this rank's slice on the device
            s_gt = torch.empty((m_gt, 3), dtype=torch.float64, device=dev)
    # one explicit (non-default) stream for everything: the library's kernels, torch's copies and the NCCL collectives are
    # ordered on it (the legacy default stream has handle 0, which the C-ABI reads as "create your own stream" — torch's
    # copies / collectives and the library's kernels would then race)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx = api.MapEvalB200(device=local_rank, rank=rank, world=world, stream=stream.cuda_stream,
                          vmd_voxel_size=cfg["vmd_voxel_size"] if cfg["awd"] else 0.0)
    # N > 1: slab layout — every rank lays out (and evaluates) only the voxel layers it owns of both clouds; the library
    # keeps the replicated layout where the scene cannot be cut (ctx.layout_active() tells which one ran)
    if world > 1 and args.layout == "slab":
        ctx.set_layout(A.ME_LAYOUT_SLAB)

    results = {}

    def one_pass(mode):
        if mode == "pinned" and world == 1:
            ctx.set_cloud_ptr(A.ME_CLOUD_EST, h_est.data_ptr(), n_est, keepalive=h_est)
            ctx.set_cloud_ptr(A.ME_CLOUD_GT, h_gt.data_ptr(), n_gt, keepalive=h_gt)
        elif mode == "pageable":
            ctx.set_cloud(A.ME_CLOUD_EST, p_est)
            ctx.set_cloud(A.ME_CLOUD_GT, p_gt)
        elif mode == "pinned":
            for h, sl, g, n, which in ((h_est, s_est, g_est, n_est, A.ME_CLOUD_EST), (h_gt, s_gt, g_gt, n_gt, A.ME_CLOUD_GT)):
                sl.copy_(h, non_blocking=True)                                   # 1/N of the cloud over this rank's PCIe link
                dist.all_gather_into_tensor(g.view(-1), sl.view(-1))             # the rest over NVLink
                ctx.set_cloud_device(which, g.data_ptr(), n, keepalive=g)
        else:
            ctx.set_cloud_device(A.ME_CLOUD_EST, d_est.data_ptr(), n_est, keepalive=d_est)
            ctx.set_cloud_device(A.ME_CLOUD_GT, d_gt.data_ptr(), n_gt, keepalive=d_gt)
        # MapEval::process() order (map_eval.cpp:56,76,85): MME, then the NN metrics, then VMD.  With host buffers
        # the GT upload (copy stream) overlaps the est lattice build + MME, which need the est cloud only.
        # the accumulators stay on the device: sweeps -> (N > 1: all-reduce in place over NCCL) -> one fetch per pass
        ctx.accum_reset()
        if cfg["mme"]:
            ctx.eval_mme_accum_device(A.ME_CLOUD_EST, cfg["nn_radius"], 10)
            if cfg["gt_mme"]:
                ctx.eval_mme_accum_device(A.ME_CLOUD_GT, cfg["nn_radius"], 5)
        ctx.eval_nn_accum_device(p)
        awd = None
        slab = world > 1 and ctx.layout_active()["layout"] == A.ME_LAYOUT_SLAB
        if cfg["awd"] and slab:
            # every rank computes the voxels of its layers; the W table is MAX-all-reduced for the SCS neighbourhoods and
            # the stage's counters / sums ride in the accumulator block
            ctx.voxel_begin(cfg["vmd_voxel_size"], 100)
            mdist.allreduce_voxel_w(ctx, dev)
            ctx.voxel_finish_accum_device(5)
        elif cfg["awd"]:
            awd = ctx.calculateVMD(cfg["vmd_voxel_size"], 100, 5)
        if world > 1:
            mdist.allreduce_block(ctx, dev)
        nn_e, nn_g, mmes = ctx.accum_fetch(want_mme=(bool(cfg["mme"]), bool(cfg["mme"] and cfg["gt_mme"])))
        if cfg["awd"] and slab:
            awd = ctx.accum_fetch_awd()
        results["layout"] = ctx.layout_active()
        results["nn"] = ctx.nn_finalize(p, nn_e, nn_g)
        results["mme"] = [ctx.mme_finalize(m, w) for m, w in zip(mmes, (A.ME_CLOUD_EST, A.ME_CLOUD_GT))]
        results["awd"] = awd
        results["n_far"] = (nn_e.n_far, nn_g.n_far)

    def timed(mode, steps, stage_acc=None):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count()
        t0 = time.time()
        ev0.record(stream)
        for _ in range(steps):
            one_pass(mode)
            if stage_acc is not None:
                for k, v in ctx.stage_times_ms().items():
                    stage_acc[k] = stage_acc.get(k, 0.0) + v
        ev1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t1 = time.time()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, ctx.launch_count() - l0, t0, t1

    torch.cuda.synchronize()      # the clouds were produced on the default stream
    for _ in range(args.warmup):
        one_pass("device")
    stage_ms = {}
    ms_dev, launches, t0, t1 = timed("device", args.steps, stage_ms)
    device_results = dict(results)      # the e2e arms below overwrite `results`
    t_last = t1
    ms_e2e = ms_page = None
    if do_e2e:
        for _ in range(min(args.warmup, 2)):
            one_pass("pinned")
        ms_e2e, _, _, t_last = timed("pinned", args.steps)
        if world == 1:
            one_pass("pageable")
            ms_page, _, _, t_last = timed("pageable", max(1, min(args.steps, 5)))
    clocks = sampler.stop(t0, t_last) if sampler else None

    if rank == 0:
        stage_ms = {k: v / args.steps for k, v in stage_ms.items()}
        value = n_est / (ms_dev * 1e-3) / 1e6
        peak, peak_src = _peaks()
        # dominant kernel: the MME radius sweep of the estimated map (stage "mme_est" = the sweep kernel + a 1-thread init).
        # algorithmic bytes per launch (SURVEY §8d): 12 B query + 12 B reference + 8 B entropy out per point of this
        # rank's query range
        lay = results.get("layout") or {}
        slab = lay.get("layout") == A.ME_LAYOUT_SLAB
        nq = lay["n_owned"][0] if slab else n_est * (rank + 1) // world - n_est * rank // world
        dom = "mme_est" if cfg["mme"] else "nn_est_to_gt"
        alg_bytes = (32.0 * nq) if cfg["mme"] else (12.0 * (nq + n_gt))
        dom_ms = stage_ms.get(dom, 0.0)
        achieved = alg_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else None
        traffic = _profile_traffic()
        same_cfg = bool(traffic) and args.config == "C3" and args.scale == 1.0 and world == 1
        roofline = {"bound": "hbm", "kernel": (traffic or {}).get("kernel_name", "mme sweep" if cfg["mme"] else "nn sweep"),
                    "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": (achieved / peak) if achieved else None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": dom_ms,
                    "traffic": traffic.get("dram_bytes_per_launch") if same_cfg else None,
                    "note": "neighbour sweep bound by issue slots and L1/L2 latency (~130 candidate tests per query served "
                            "from cache / shared memory); the HBM fraction is small by construction (SURVEY §8d, DESIGN §3)"}
        # the resource that actually binds the sweep: warp-instruction issue slots (4 schedulers x 1 instruction per
        # clock per SM).  Instruction, candidate-test and accepted-pair counts per launch come from the committed ncu
        # capture of this kernel on this config (profiles/roofline_traffic.json); the time is this run's.
        binding = None
        if same_cfg and dom_ms > 0 and traffic.get("warp_inst_per_launch"):
            sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
            issue_peak = 148 * 4 * sm_mhz * 1e6
            wi = float(traffic["warp_inst_per_launch"])
            binding = {"resource": "warp-instruction issue slots", "achieved": wi / (dom_ms * 1e-3), "peak": issue_peak,
                       "unit": "warp-inst/s", "frac": wi / (dom_ms * 1e-3) / issue_peak,
                       "candidate_tests_per_s": float(traffic.get("candidate_tests_per_launch", 0)) / (dom_ms * 1e-3),
                       "accepted_pairs_per_s": float(traffic.get("accepted_pairs_per_launch", 0)) / (dom_ms * 1e-3),
                       "thread_inst_per_warp_inst": traffic.get("thread_inst_per_warp_inst"),
                       "source": traffic.get("source")}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            from oracle import oracle as O  # noqa: F401
            threads = _host_threads()
            s_est, s_gt, s_cfg, s_scale = _cpu_sample(args.config)
            dt = _cpu_pass(s_est, s_gt, s_cfg, threads)
            cpu = {"value": len(s_est) / dt / 1e6, "unit": UNIT, "cores": threads, "kind": "port", "voxel_hash": VOXEL_HASH_NOTE,
                   "sample": f"{args.config} at scale {s_scale:g} ({len(s_est)} est vs {len(s_gt)} gt points, same "
                             f"density), one full pass in {dt:.1f} s, all-cores mode"}
        nn = results["nn"]
        d2h = (2 * C.sizeof(A.me_nn_accum) + C.sizeof(A.me_mme_accum) * len(results["mme"]) + C.sizeof(A.me_awd_result))
        e2e = None
        if ms_e2e:
            e2e = {"value": n_est / (ms_e2e * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms_e2e,
                   "h2d_bytes_per_step": 24 * (m_est + m_gt) if world > 1 else 24 * (n_est + n_gt),
                   "d2h_bytes_per_step": d2h,
                   "host_memory": "pinned" if world == 1 else
                   f"pinned; each rank uploads 1/{world} of both clouds, slices all-gathered over NVLink (NCCL) inside the timed region"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{args.config}: {synth.CONFIGS[args.config]['desc']}", "n_est": n_est,
                       "n_gt": n_gt, "tau": cfg["tau"], "icp_max_distance": 1.0, "nn_radius": cfg["nn_radius"],
                       "vmd_voxel_size": cfg["vmd_voxel_size"], "mme_gt": bool(cfg["gt_mme"]),
                       "generated": gen,
                       "planning": "the context remembers the lattice plan (refined cell edge, slab cut) of a cloud pair: passes "
                                   "after the first plan in one step instead of 2-3 histogram passes; the lattices themselves "
                                   "are rebuilt from the points every pass",
                       "parallelism": (f"slab layout x{world}: voxel layers along {'xyz'[lay.get('axis', 0)]} owned per rank, lattice builds, "
                                       f"sweeps and voxel stage sharded; rank 0 lays out {lay['n_laid_out'][0]} + {lay['n_laid_out'][1]} "
                                       f"points and evaluates {lay['n_owned'][0]} + {lay['n_owned'][1]}") if slab else
                                      f"query-range shard x{world}, lattices replicated",
                       "l2": f"inputs per pass ({24 * (n_est + n_gt) / 1e6:.0f} MB of fp64 clouds, {48 * (n_est + n_gt) / 1e6:.0f} MB of "
                             "sorted records and fp32 screening copies) exceed the 126 MB L2 several times over; no flush needed"},
            "e2e": e2e,
            "gpu_launches": launches,
            "roofline": roofline,
            "cpu_baseline": cpu,
            "clocks": clocks,
            "stage_ms": stage_ms,
            "check": {"AC_rmse": list(nn.est_to_gt.rmse), "n_inlier": list(nn.est_to_gt.n_inlier),
                      "n_inlier_gt_to_est": list(nn.gt_to_est.n_inlier), "n_corr": [nn.est_to_gt.n_corr, nn.gt_to_est.n_corr],
                      "full_cd": nn.full_cd, "mme": [m.mme for m in results["mme"]],
                      "mme_n_valid": [m.n_valid for m in results["mme"]],
                      "awd": results["awd"].awd if results["awd"] else None,
                      "scs": results["awd"].scs if results["awd"] else None,
                      "awd_n_pairs": results["awd"].n_pairs if results["awd"] else None, "n_far": list(results["n_far"])},
        }
        if binding:
            line["roofline_binding"] = binding
        if ms_page:
            line["e2e_pageable"] = {"value": n_est / (ms_page * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms_page,
                                    "h2d_bytes_per_step": 24 * (n_est + n_gt), "d2h_bytes_per_step": d2h,
                                    "host_memory": "pageable (plain numpy arrays handed to me_set_cloud, the way a "
                                                   "std::vector<Eigen::Vector3d> caller does)"}
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
        if args.dump_outputs:
            _dump_outputs(args.dump_outputs, device_results)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
