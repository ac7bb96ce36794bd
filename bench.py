#!/usr/bin/env python
"""Benchmark of the temporal articulation optimizer hot path (contract: task spec §④).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c3_shard|c4|c4_trans]
    python bench.py --impl reference ...     # the CPU oracle port on the host cores
    torchrun ... bench.py --gpus N ...       # one rank per GPU: the workload's videos are sharded over
                                             # the ranks in contiguous blocks (strong scaling)
    python bench.py --dump-outputs DIR ...   # also write the last timed step's outputs as DIR/<name>.npy

The headline workload is BASELINE.json configs[2]: 256 videos x 8 tracks x 120 frames, 180-angle grid —
the configuration the metric (track-frames x angles / s at 1/2/4/8 B200) is quoted on; it fits one GPU
(9.4 GB of packed masks + 14 GB of projected masks), so N=1 runs all of it and N ranks run 256/N videos
each (the reference's SLURM split, tools/opt_arti.py:116-123).

A *step* is one scoring pass over the workload: per track one source frame is unprojected, moved by every
candidate transform, re-projected and scored against every frame of the track (k_unproject, k_project,
scoring kernel, k_finalize), and the fixed-size per-track-frame records are gathered to every rank.
``value`` counts track-frame x candidate IoU evaluations per second with all inputs resident in HBM;
``e2e`` is the same metric through the public API (``dist.optimize_videos_sharded`` ->
``optimize_videos``) with HOST fp32 masks (H2D, packing, every device pass, D2H and the record gather inside
the timed region).  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "track_frames_x_angles_per_sec"
UNIT = "track-frame*angle IoU evaluations/s"
# the clip both arms are quoted on beside their own samples: the reference arm times the CPU port on it,
# the GPU arm's e2e also runs it through the public API (`e2e.reference_sample`)
REF_SAMPLE = (1, 40)            # (tracks, frames) of the workload's clip shape and grids
# --dump-outputs: bytes of all files together; the device pass gets 3/4, the e2e leg 1/4
DUMP_BYTES = 64 * 10 ** 6
DUMP_SEED = 2020
NPY_HEADER = 128                # bytes of a .npy header of these small-rank arrays


def dump_arrays(arrays, budget, seed=DUMP_SEED):
    """name -> tensor  ->  name -> float32 / float64 numpy array, all of them together within ``budget`` bytes.
    Integer arrays become float64 (exact for 32-bit values); floating arrays keep float32 / float64.  An array
    larger than its share of the budget is replaced by a seeded sample of its rows (leading dimension) whose
    sorted indices are stored as ``<name>_rows``; the sample depends only on the shape, so two runs with the same
    arguments dump the same rows.  Each file is counted with NPY_HEADER bytes of header."""
    out = {}
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    for i, (name, t) in enumerate(items):
        share = budget // (len(items) - i) - NPY_HEADER
        t = t.detach()
        dtype = torch.float32 if t.dtype in (torch.float16, torch.bfloat16, torch.float32) else torch.float64
        n = t.shape[0] if t.dim() else 1
        row = (t[0].numel() if t.dim() and n else 1) * (4 if dtype == torch.float32 else 8)
        if n * row > share:
            k = min(n, max(1, (share - NPY_HEADER) // (row + 8)))
            rows = np.sort(np.random.default_rng(seed).choice(n, size=k, replace=False))
            out[name + "_rows"] = rows.astype(np.float64)
            budget -= out[name + "_rows"].nbytes + NPY_HEADER
            t = t.index_select(0, torch.from_numpy(rows).to(t.device))
        out[name] = t.to(dtype).cpu().numpy()
        budget -= out[name].nbytes + NPY_HEADER
    return out


def write_dump(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region: the sampler is started ahead of the
    warm-up (nvidia-smi needs a few hundred ms to deliver its first line) and every line carries its own
    timestamp, so only the samples that fall inside the timed region are reported."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float | None = None, t1: float | None = None):
        """``t0``, ``t1``: time.time() at the start / end of the timed region."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        import datetime
        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for seen, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 10:
                continue
            try:
                when = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((when, float(f[2]), float(f[3]), [nm for nm, val in zip(names, f[6:10]) if val.lower().startswith("active")]))
            except ValueError:
                continue
        inside = [r for r in rows if t0 is not None and t0 - 0.02 <= r[0] <= t1 + 0.02]
        where = "inside the timed region"
        if len(inside) < 2 and rows and t0 is not None:
            # a timed region shorter than two sampling periods: the samples nearest to it (same load: warm-up
            # steps before, the split steps after)
            inside = sorted(rows, key=lambda r: abs(r[0] - 0.5 * (t0 + t1)))[:4]
            where = "nearest to the timed region (shorter than two sampling periods)"
        if t0 is None:
            inside, where = rows, "whole run"
        sm = [r[1] for r in inside]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max((r[2] for r in inside), default=None),
                "samples": len(sm), "sampled": where, "reasons": sorted({x for r in inside for x in r[3]})}


# --------------------------------------------------------------------------
# CPU oracle port timing (cpu_baseline / --impl reference)
# --------------------------------------------------------------------------
def _oracle_cfg(cfg):
    from oracle import restated
    return restated.OracleConfig(height=cfg.height, width=cfg.width, focal_length=cfg.focal_length,
                                 rot_cluster_grid=cfg.rot_cluster_grid, rot_final_grid=cfg.rot_final_grid,
                                 trans_grid=cfg.trans_grid)


def _count_units(trace, cfg):
    n = 0
    for step in trace:
        if step["kind"] == "trans":
            a = len(cfg.trans_grid)
        else:
            a = len(cfg.rot_cluster_grid) if step["phase"] == "cluster" else len(cfg.rot_final_grid)
        n += a * len(step["visits"])
    return n


def run_oracle_sample(wl, seed, tracks, frames):
    """One run of the CPU port on a (tracks x frames) sample of the workload -> (seconds, units)."""
    from articulation3d_b200 import workloads
    from oracle import restated
    preds, cfg = workloads.make_clip(wl, seed, tracks=tracks, frames=frames)
    random.seed(seed)
    t0 = time.perf_counter()
    planes = restated.track_planes(preds)
    trace = []
    restated.optimize_planes(preds, planes, "3dc", cfg=_oracle_cfg(cfg), trace=trace)
    dt = time.perf_counter() - t0
    return dt, _count_units(trace, cfg)


def pick_sample(wl, budget_s: float):
    """(tracks, frames) sample of the workload's clip for the CPU port: REF_SAMPLE when one run of it fits
    ``budget_s`` on this host (the usual case — both arms then quote the same clip), else the largest
    smaller one that does."""
    dt, units = run_oracle_sample(wl, 2020, 1, 24)            # calibration (also warms torch)
    rate = max(units, 1) / dt
    ladder = [REF_SAMPLE, (1, 32), (1, 24)]
    cand = len(wl.cfg().rot_cluster_grid)
    final = len(wl.cfg().rot_final_grid)
    for tr, fr in ladder:
        est_units = tr * (2 * fr * cand + fr * final)         # ~2T visits in the cluster rounds + T final
        if est_units / rate <= budget_s:
            return tr, fr, rate
    return 1, 24, rate


def reference_arm(args, wl):
    """--impl reference: the reference's CPU implementation (oracle port) on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    total = args.steps + args.warmup
    tr, fr, _ = pick_sample(wl, budget_s=max(2.0, 200.0 / max(total, 1)))
    for _ in range(args.warmup):
        run_oracle_sample(wl, 2020, tr, fr)
    secs, units = 0.0, 0
    for _ in range(args.steps):
        dt, u = run_oracle_sample(wl, 2020, tr, fr)
        secs += dt
        units += u
    value = units / secs
    sample = (f"{tr} track(s) x {fr} frames of the {wl.name} clip shape ({len(wl.cfg().rot_cluster_grid)}/"
              f"{len(wl.cfg().rot_final_grid)}-candidate grids, {wl.width}x{wl.height}), full "
              f"track_planes + optimize_planes('3dc') incl. cluster rounds, seed 2020")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(args.steps, 1),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32 popcount / fp32+fp64 geometry", "data": "synthetic",
        "config": {"workload": wl.description, "name": wl.name, "sample": sample,
                   "same_clip_as": "e2e.reference_sample of the b200 arm" if (tr, fr) == REF_SAMPLE else None,
                   "what": "oracle/restated.py: the CPU restatement of the reference's algorithm (torch CPU ops, all "
                           "host threads); /root/reference does not exist on the GPU box and its detectron2 / pytorch3d "
                           "dependencies are not installable, so the unmodified reference cannot be the thing timed"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------
def _committed(name, wl_name, kernel_key):
    """A number of a committed ncu capture (profiles/<name>.json), labelled with its source: these are
    NOT measured by this run (ncu cannot run inside a timed benchmark)."""
    path = os.path.join(ROOT, "profiles", name + ".json")
    if not os.path.exists(path):
        return None
    with open(path) as f:
        d = json.load(f)
    v = d.get(wl_name)
    if v is None:
        return None
    if kernel_key is not None:
        v = v.get(kernel_key)
        if v is None:
            return None
    return {"value": v, "source": f"committed ncu capture, profiles/{name}.json ({d.get('_source', '')})"}


def measure_pass(wl, video_ids, steps, warmup, dev, rank, world, dist, sample_clocks=True, gather=True, streams=1,
                 dump=None):
    """Device-resident scoring passes over this rank's videos of the workload: K timed steps with CUDA
    events on the launching stream -> dict(value, ms, roofline, ...).  ``value`` is the whole job: the units
    of all ranks over the slowest rank's step time.  ``dump`` (a dict) receives the PassResult of the last
    timed step as ``pass_*`` arrays (dump_arrays)."""
    from articulation3d_b200 import engine, workloads

    inp = workloads.build_pass(wl, seed0=2020, device=dev, video_ids=video_ids)
    gather = gather and world > 1
    packed_bytes = inp.pool.bits.numel() * 4
    l2_bytes = 126 * 2 ** 20
    flush = None if packed_bytes > 2 * l2_bytes else torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    # Steps are independent passes; ``streams`` = 2 lets consecutive steps alternate between two streams, each
    # with its own set of pass buffers, so that the last, partly filled wave of step k overlaps step k+1
    # (an experiment switch: see --streams).  Small workloads (L2 flush between steps) always use one.
    n_streams = 1 if flush is not None else max(1, min(2, streams))
    lanes = [torch.cuda.Stream(device=dev) for _ in range(n_streams)] if n_streams > 1 else [torch.cuda.current_stream()]
    # two sets of pass buffers also when ranks exchange results: the gather of step k reads the result block of
    # step k in place while step k+1 writes the other set (no staging copy in the step)
    wss = [engine.Workspace(dev) for _ in range(2 if (gather or n_streams > 1) else 1)]
    ws = wss[0]
    # multi-GPU: the only exchange of the path is the gather of the fixed-size per-track-frame records
    # {angle_id, inter, union} (12 B each): ONE all_gather_into_tensor per step on a side stream,
    # double-buffered, so the collective of step k overlaps the kernels of step k+1.
    n_rec = 3 * inp.dbatch.n_tgt_total
    gathered, comm_stream, comm_done = None, None, [None, None]
    if gather:
        t = torch.tensor([n_rec], device=dev, dtype=torch.int64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        n_max = int(t.item())                                   # ranks hold equal shards when N divides 256
        send = [torch.zeros(n_max, dtype=torch.int32, device=dev) for _ in range(2)] if n_max != n_rec else None
        gathered = [torch.zeros(world * n_max, dtype=torch.int32, device=dev) for _ in range(2)]
        comm_stream = torch.cuda.Stream(device=dev)
    step_no = [0]

    def one_step(evs=None, split=False):
        """One pass through the C ABI.  split=False: a3d_pass, the call the package makes, on the step's lane.
        split=True: a3d_project | a3d_score on the current stream with an event between the two launch groups,
        for the per-kernel durations of the roofline."""
        if split:
            if flush is not None:
                flush.zero_()
            evs[0].record()
            res = _run_split(engine, inp, ws, evs)
            evs[2].record()
            return res
        b = step_no[0] & 1 if len(wss) > 1 else 0
        lane = lanes[step_no[0] % len(lanes)]
        with torch.cuda.stream(lane):
            if flush is not None:
                flush.zero_()
            if evs:
                evs[0].record()
            if gather and comm_done[b] is not None:
                lane.wait_event(comm_done[b])                         # buffer set b free again
            res = engine.run_pass(inp.cfg, inp.pool, inp.dbatch, wss[b])
            if gather:
                rec = res.block[:3].reshape(-1)               # the three rows are contiguous in the result block
                if send is not None:
                    send[b][:n_rec].copy_(rec)
                    rec = send[b]
                ready = torch.cuda.Event()
                ready.record()
                with torch.cuda.stream(comm_stream):
                    comm_stream.wait_event(ready)
                    dist.all_gather_into_tensor(gathered[b], rec)
                    comm_done[b] = torch.cuda.Event(enable_timing=True)
                    comm_done[b].record()
            if evs:
                evs[2].record()
        step_no[0] += 1
        return res

    sampler = ClockSampler(dev.index).start() if (rank == 0 and sample_clocks) else None
    for _ in range(max(warmup, 3)):
        one_step()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    events = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    main = torch.cuda.current_stream()
    wall0, region0 = time.perf_counter(), time.time()
    # Let the host run ahead of the device: the GPU spins ~40 ms while all K steps are
    # enqueued, so the timed interval below contains kernel time only, never launch gaps.
    torch.cuda._sleep(int(0.04 * 1.9e9))
    t_begin.record()
    for lane in lanes:
        lane.wait_event(t_begin)
    for k in range(steps):
        last = one_step(events[k])
    for lane in lanes:                                  # join: the timed region ends when every lane has drained
        done = torch.cuda.Event()
        done.record(lane)
        main.wait_event(done)
    if gather:
        main.wait_event(comm_done[(step_no[0] - 1) & 1])          # ... and the last gather has landed
        if steps > 1:
            main.wait_event(comm_done[(step_no[0] - 2) & 1])
    t_end.record()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    wall, region1 = time.perf_counter() - wall0, time.time()
    clocks = sampler.stop(region0, region1) if sampler else None
    if dump is not None:                                # before the split steps below overwrite the workspace
        dump.update(dump_arrays({"pass_" + f: getattr(last, f) for f in (
            "best_cand", "best_inter", "best_union", "best_iou", "proj_bits", "proj_popc", "proj_bbox")},
            DUMP_BYTES * 3 // 4))
    del last                                            # views of the workspace, released with it below
    # the timed K steps: one device interval from the first launch to the last lane / gather draining
    # (with one lane and an L2 flush between steps: the sum of the per-step intervals, which leave the flush out)
    if flush is not None:
        t_step = sum(e[0].elapsed_time(e[2]) for e in events) / steps
    else:
        t_step = t_begin.elapsed_time(t_end) / steps
    # the same K steps again as a3d_project | a3d_score, for the kernel durations of the roofline
    split_events = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    torch.cuda._sleep(int(0.04 * 1.9e9))
    for k in range(steps):
        one_step(split_events[k], split=True)
    torch.cuda.synchronize()
    # medians: one disturbed step (a clock dip while the split steps run) must not move the kernel durations
    t_proj = statistics.median(e[0].elapsed_time(e[1]) for e in split_events)
    t_score = statistics.median(e[1].elapsed_time(e[2]) for e in split_events)
    t_split = statistics.median(e[0].elapsed_time(e[2]) for e in split_events)
    units_all = inp.units
    per_rank_ms = [t_step]
    if world > 1:
        t = torch.tensor([t_step, t_proj, t_score], device=dev, dtype=torch.float64)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank_ms = [float(x[0]) for x in allt]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_step, t_proj, t_score = t.tolist()
        u = torch.tensor([inp.units], device=dev, dtype=torch.int64)
        dist.all_reduce(u)
        units_all = int(u.item())
    value = units_all / (t_step * 1e-3)

    # ---- roofline of the dominant kernel (this rank's launch) ---------------------------
    peak, peak_src = _peaks()
    alg = wl.alg_bytes_per_pass() * len(video_ids) // wl.videos
    proj_dom = t_proj >= t_score
    dom, t_alone = ("a3d_project (k_unproject + k_project)", t_proj) if proj_dom else \
                   ("a3d_score (scoring kernel + k_finalize)", t_score)
    # the dominant kernel's duration inside the timed steps: its share of a step issued as two calls, applied to
    # the timed step (the two agree to ~1 % when nothing disturbs the split steps; the share is what the ncu
    # launch list under profiles/ has to confirm)
    t_dom = t_step * t_alone / t_split
    achieved = alg / (t_dom * 1e-3) / 1e9
    cap_name = wl.name if world == 1 else f"{wl.name}/{world}"
    traffic = _committed("traffic", cap_name, "k_project" if proj_dom else "k_score")
    pipes = _committed("pipes", cap_name, None)
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic["value"] if traffic else None,
                "traffic_source": traffic["source"] if traffic else None, "peak_source": peak_src,
                "alg_bytes_per_launch": alg, "kernel_ms": t_dom,
                "kernels_ms": {"project": t_proj, "score": t_score, "step_two_calls": t_split, "step": t_step,
                               "how": "project / score / step_two_calls: medians over the K steps issued alone as "
                                      "a3d_project | a3d_score; kernel_ms = step x share of the dominant call"},
                "pipes_pct_of_peak": pipes["value"] if pipes else None,
                "pipes_source": pipes["source"] if pipes else None,
                "note": "bit-packed masks make the pass ALU-bound (fp32 splat / AND+POPC), not HBM-bound; "
                        "achieved = SURVEY 8d algorithmic bytes of this rank's launch / dominant-kernel time"}
    n_jobs = inp.dbatch.n_jobs
    del inp, ws, wss
    torch.cuda.empty_cache()
    return {"value": value, "ms_per_step": t_step, "roofline": roofline, "units_per_step": units_all,
            "units_per_step_per_gpu": units_all // world, "jobs_per_gpu": n_jobs, "per_rank_ms": per_rank_ms,
            "packed_mask_bytes_per_gpu": packed_bytes, "streams": n_streams,
            "l2": "flushed between steps (256 MiB write)" if flush is not None else "inputs exceed L2",
            "clocks": clocks, "wall_s": wall}


def gpu_arm(args, wl):
    from articulation3d_b200 import dist as a3d_dist
    from articulation3d_b200 import workloads

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the hot path has no CPU fallback "
                         "(use --impl reference for the CPU oracle port)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # Intra-op threads of the host side (small float64 array work of the public API).  torchrun's OMP_NUM_THREADS=1
    # per rank is kept: with cores // world threads per rank (round 2's first choice) the idle OpenMP workers of
    # the ranks spin on every core of the box and starve the upload / preparation / NCCL threads — 612 ms per e2e
    # step at N = 2 against 167 ms with one thread (gpurun_out/bench_n2_t1.txt); at N = 1 one, two, four and sixteen
    # threads measure the same (the step is bound by the H2D copy), four is taken.
    torch.set_num_threads(1 if world > 1 else min(4, os.cpu_count() or 1))
    if os.environ.get("A3D_BENCH_THREADS"):              # experiment switch: intra-op threads of the host side
        torch.set_num_threads(int(os.environ["A3D_BENCH_THREADS"]))
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)

    mine = list(a3d_dist.shard_range(wl.videos, rank, world))
    dump = {} if args.dump_outputs and rank == 0 else None
    m = measure_pass(wl, mine, args.steps, args.warmup, dev, rank, world, dist, streams=args.streams, dump=dump)
    # ---- e2e through the public API with host buffers, sharded like the device-resident pass -----
    e2e = _e2e(wl, dev, rank, world, dist, steps=args.steps, videos_per_rank=args.e2e_videos, dump=dump)
    if dump is not None:
        write_dump(args.dump_outputs, dump)

    line = None
    if rank == 0:
        extras = {}
        if world == 1 and args.extras:
            # configs[1] (one video, 4 tracks x 60 frames, 90 candidates): a 57 us launch-latency case
            wc = workloads.WORKLOADS["c2"]
            mc = measure_pass(wc, [0], args.steps, 3, dev, 0, 1, None, sample_clocks=False)
            extras["c2"] = {"workload": wc.description, "value": mc["value"], "unit": UNIT,
                            "ms_per_step": mc["ms_per_step"], "units_per_step": mc["units_per_step"], "l2": mc["l2"],
                            "roofline": mc["roofline"]}
            extras["pack"] = _pack_stream(dev)
        # ---- CPU port on a bounded sample (N=1 only) -----------------------------------
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            tr, fr, _ = pick_sample(wl, budget_s=25.0)
            dt, u = run_oracle_sample(wl, 2020, tr, fr)
            cpu = {"value": u / dt, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"{tr} track(s) x {fr} frames of the {wl.name} clip shape, track_planes + "
                             f"optimize_planes('3dc'), {dt:.1f} s"}
        line = {
            "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": m["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u32 popcount / fp32+fp64 geometry",
            "data": "synthetic",
            "config": {"workload": wl.description, "name": wl.name, "videos_total": wl.videos,
                       "videos_per_gpu": len(mine), "units_per_step": m["units_per_step"],
                       "units_per_step_per_gpu": m["units_per_step_per_gpu"], "jobs_per_gpu": m["jobs_per_gpu"],
                       "packed_mask_bytes_per_gpu": m["packed_mask_bytes_per_gpu"], "l2": m["l2"],
                       "per_rank_ms_per_step": m["per_rank_ms"],
                       "step": "one a3d_pass call (k_unproject, k_project, scoring kernel, k_finalize) on device-resident "
                               "inputs + the record gather; consecutive (independent) steps alternate between "
                               f"{m['streams']} stream(s) with their own pass buffers; timed as ONE device interval over the K "
                               "steps; roofline.kernels_ms from the same K steps issued alone as a3d_project | a3d_score",
                       "kernels": "chosen by the library from the grid: projection = homography filter with proven "
                                  "truncation (reference chain for the unproven pairs); scoring = tcgen05 kind::i8 "
                                  "contraction of the bit masks; identical results to the reference chain / AND+POPC",
                       "parallelism": (f"videos sharded x{world} in contiguous blocks (same total at every N); per step "
                                       f"ONE all_gather_into_tensor of 12 B/track-frame records on a side stream "
                                       f"(overlaps the next step)") if world > 1 else "single GPU, all videos"},
            "roofline": m["roofline"], "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": 4 * args.steps, "clocks": m["clocks"], "wall_s": m["wall_s"], "extras": extras,
        }
        print(json.dumps(line), flush=True)
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return line


def _pack_stream(dev, n_masks=1024, H=480, W=640, iters=5):
    """The one pure HBM stream of the path: fp32 (n,H,W) -> packed bits (a3d_pack_masks), timed
    alone with CUDA events; input (1.26 GB) exceeds L2.  Reported against the measured HBM peak."""
    from articulation3d_b200 import _lib
    lib = _lib.load()
    src = (torch.rand(n_masks, H, W, device=dev, generator=torch.Generator(dev).manual_seed(2020)) > 0.7).float()
    pitch = _lib.pitch_words(W)
    bits = torch.empty(n_masks, H, pitch, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * iters)]
    for k in range(3 + iters):
        if k >= 3:
            ev[2 * (k - 3)].record()
        _lib.check(lib.a3d_pack_masks(src.data_ptr(), _lib.A3D_F32, n_masks, H, W, 0.5, bits.data_ptr(), None, stream),
                   "a3d_pack_masks")
        if k >= 3:
            ev[2 * (k - 3) + 1].record()
    torch.cuda.synchronize()
    ms = min(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(iters))
    nbytes = src.numel() * 4 + bits.numel() * 4
    peak, src_name = _peaks()
    gbs = nbytes / (ms * 1e-3) / 1e9
    return {"kernel": "a3d_pack_masks (k_pack_vec<float>)", "bytes": nbytes, "ms": ms, "achieved": gbs, "unit": "GB/s",
            "peak": peak, "frac": gbs / peak, "peak_source": src_name, "bound": "hbm"}


def _run_split(engine, inp, ws, evs):
    """engine.run_pass with an event between a3d_project and a3d_score."""
    import ctypes as C

    from articulation3d_b200 import _lib
    lib = _lib.load()
    cfg, pool, db = inp.cfg, inp.pool, inp.dbatch
    H, W = cfg.height, cfg.width
    pitch = _lib.pitch_words(W)
    nc, nt = db.n_cand_total, db.n_tgt_total
    proj_bits, proj_popc, proj_bbox = ws.get_proj(nc, H, pitch)
    pcd_ws = ws.get("pcd_ws", (max(_lib.PCD_PLANES * db.pcd_total, 32),), torch.float32)
    pcd_count = ws.get("pcd_count", (db.n_jobs + 1,), torch.int32)
    hom_ws = ws.get("hom_ws", (max(nc, 1), _lib.HOM_FLOATS), torch.float32)
    key_ws = ws.get("key_ws", (nt,), torch.int64)
    outs = [ws.get(n, (nt,), dt) for n, dt in (("best_cand", torch.int32), ("best_inter", torch.int32),
                                               ("best_union", torch.int32), ("best_iou", torch.float32))]
    cam = engine.camera_struct(cfg)
    stream = torch.cuda.current_stream().cuda_stream
    tile, tmap = db.tile_plan(cfg)
    tmap_ptr, n_tiles = (tmap.data_ptr(), int(tmap.shape[0])) if tmap is not None else (None, 0)
    _lib.check(lib.a3d_project(C.byref(cam), db.jobs.data_ptr(), db.n_jobs, db.max_cand, tile,
                               pool.source_bits.data_ptr(), pool.source_bbox.data_ptr(), db.xform.data_ptr(),
                               pcd_ws.data_ptr(), pcd_count.data_ptr(), hom_ws.data_ptr(), tmap_ptr, n_tiles,
                               proj_bits.data_ptr(), proj_popc.data_ptr(), proj_bbox.data_ptr(),
                               engine.default_out_mode(), stream),
               "a3d_project")
    if evs:
        evs[1].record()
    _lib.check(lib.a3d_score(H, W, db.jobs.data_ptr(), db.n_jobs, db.max_tgt, db.max_cand, nt,
                             len(pool), nc, pool.bits.data_ptr(), pool.popc.data_ptr(), pool.bbox.data_ptr(),
                             db.tgt_index.data_ptr(), proj_bits.data_ptr(), proj_popc.data_ptr(),
                             proj_bbox.data_ptr(), key_ws.data_ptr(), None, outs[0].data_ptr(),
                             outs[1].data_ptr(), outs[2].data_ptr(), outs[3].data_ptr(), stream), "a3d_score")
    return engine.PassResult(outs[0], outs[1], outs[2], outs[3], proj_bits, proj_popc, proj_bbox, None,
                             rows_only=engine.default_out_mode() == _lib.OUT_BBOX_ROWS)


def _host_clip(wl, seed, dev, tracks=None, frames=None, pin=True):
    """One clip of the workload's shape as HOST predictions: rendered on the device (the CPU renderer takes
    seconds per track), masks moved to pinned host memory."""
    from articulation3d_b200 import synth
    cfg = wl.cfg()
    tracks, frames = tracks or wl.tracks, frames or wl.frames
    preds, _ = synth.make_video(seed, tracks, frames, cfg, kinds=[synth.KIND_ROT] * tracks, device=dev)
    for p in preds:
        p.pred_masks = p.pred_masks.cpu().pin_memory() if pin else p.pred_masks.cpu()
    torch.cuda.synchronize()
    return preds, cfg


def _e2e(wl, dev, rank, world, dist, steps, videos_per_rank, dump=None):
    """Public API, host buffers: ``videos_per_rank`` clips of the workload's shape per rank (fp32 masks in
    pinned host memory) -> dist.optimize_videos_sharded (track_planes, H2D, packing, every device pass, D2H,
    write-back, record gather).  Timed with the wall clock between barriers, max over ranks.  ``dump`` (a dict)
    receives what the last timed step returned as ``e2e_*`` arrays: this rank's output instances of all frames
    in video order (scores, planes, axes) and the gathered frame / track records."""
    from articulation3d_b200 import dist as a3d_dist
    from articulation3d_b200 import opt_utils

    n_videos = videos_per_rank * world
    mine = list(a3d_dist.shard_range(n_videos, rank, world))
    clips = {v: _host_clip(wl, 2020 + v, dev)[0] for v in mine}
    cfg = wl.cfg()
    seeds = [2020 + v for v in range(n_videos)]
    saved = {v: [(p.pred_tran_axis.clone(), p.pred_rot_axis.clone(), p.pred_planes.clone()) for p in clips[v]]
             for v in mine}
    # the clips are ~10^5 long-lived Python objects: keep the cyclic collector's full passes (tens of ms, at
    # allocation-count-dependent moments) off them, as a long-running host process would
    import gc
    gc.collect()
    gc.freeze()

    def restore():          # optimize_planes rebinds / mutates the axis fields of its inputs
        for v in mine:
            for p, (ta, ra, pl) in zip(clips[v], saved[v]):
                p.pred_tran_axis, p.pred_rot_axis, p.pred_planes = ta.clone(), ra.clone(), pl.clone()

    def run():
        stats = opt_utils.Stats()

        def fn(videos, sds, cfg=None, device=None):
            return opt_utils.optimize_videos(videos, sds, cfg=cfg, device=device, stats=stats)
        t0 = time.perf_counter()
        # remote videos are never touched by this rank: placeholders keep the global numbering
        # (preds, None): optimize_videos runs track_planes itself, video by video inside its upload pipeline
        vids = [(clips[v], None) for v in range(n_videos)] if world == 1 else \
               [(clips[v], None) if v in clips else (None, None) for v in range(n_videos)]
        outs, ids, fr, tr = a3d_dist.optimize_videos_sharded(vids, seeds, cfg=cfg, device=dev, optimize_fn=fn)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        return dt, stats, fr, tr, outs

    per_rank = []

    def synced_run():
        if dist:
            dist.barrier()
        dt, st, fr, tr, outs = run()
        if dist:
            t = torch.zeros(world, device=dev, dtype=torch.float64)
            t[rank] = dt
            dist.all_reduce(t)
            per_rank.append([round(1e3 * float(x), 1) for x in t.tolist()])
            dt = float(t.max().item())
        return dt, st, fr, tr, outs

    synced_run()
    restore()
    secs, units, h2d, d2h, passes, sched = 0.0, 0, 0, 0, 0, ""
    n_frame_rec = n_track_rec = 0
    each = []
    for k in range(steps):
        dt, st, fr, tr, outs = synced_run()
        if dump is not None and k == steps - 1:
            frames = [p for preds in outs for p in preds]
            dump.update(dump_arrays({
                "e2e_scores": torch.from_numpy(np.concatenate([np.asarray(p.scores, dtype=np.float64).reshape(-1)
                                                               for p in frames])),
                "e2e_pred_planes": torch.cat([p.pred_planes for p in frames]),
                "e2e_pred_rot_axis": torch.cat([p.pred_rot_axis for p in frames]),
                "e2e_pred_tran_axis": torch.cat([p.pred_tran_axis for p in frames]),
                "e2e_frame_records": fr, "e2e_track_records": tr}, DUMP_BYTES // 4))
        secs += dt
        each.append(round(1e3 * dt, 2))
        u = torch.tensor([st.units_visited, st.h2d_bytes, st.d2h_bytes], device=dev, dtype=torch.int64)
        if dist:
            dist.all_reduce(u)
        units += int(u[0])
        h2d += int(u[1])
        d2h += int(u[2])
        passes += st.passes
        sched = st.schedule
        n_frame_rec, n_track_rec = int(fr.shape[0]), int(tr.shape[0])
        restore()
    out = {"value": units / secs, "unit": UNIT, "h2d_bytes_per_step": h2d // steps,
           "d2h_bytes_per_step": d2h // steps, "ms_per_step": 1e3 * secs / steps, "ms_each_step": each,
           "api": f"dist.optimize_videos_sharded -> optimize_videos('3dc') on {n_videos} video(s) of the {wl.name} "
                  f"clip shape ({wl.tracks} tracks x {wl.frames} frames, {videos_per_rank} per GPU), fp32 host masks "
                  f"(pinned); timed: track_planes (inside the batch call, pipelined with the uploads), H2D, packing, all device passes, D2H, write-back, record gather; "
                  f"units = visited (frame, candidate) pairs as the reference counts them",
           "videos": n_videos, "schedule": sched, "device_passes_per_step_rank0": passes // steps,
           "gathered_records": {"track_frames": n_frame_rec, "tracks": n_track_rec}}
    if per_rank:
        out["ms_each_step_per_rank"] = per_rank[1:]
    # SURVEY test tier T5 on the real thing: the records every rank received must equal what ONE GPU computes.
    # Videos are independent (each draws from its own seeded generator), so rank 0 re-runs, alone and untimed,
    # its own videos plus the first video of every other rank (rendered from its seed) and compares their rows.
    if world > 1:
        ok = torch.zeros(1, dtype=torch.int32, device=dev)
        if rank == 0:
            ids = sorted(set(mine) | {a3d_dist.shard_range(n_videos, r, world)[0] for r in range(world)})
            some = {v: (clips[v] if v in clips else _host_clip(wl, 2020 + v, dev, pin=False)[0]) for v in ids}
            vids = [(some[v], opt_utils.track_planes(some[v], cfg)) for v in ids]
            opt_utils.optimize_videos(vids, [seeds[v] for v in ids], cfg=cfg, device=dev)
            fr1, tr1 = a3d_dist.pack_records(ids, [pl for _, pl in vids])
            idt = torch.tensor(ids, dtype=torch.int32)
            frc, trc = fr.cpu(), tr.cpu()
            ok[0] = int(torch.equal(fr1, frc[torch.isin(frc[:, 0], idt)]) and torch.equal(tr1, trc[torch.isin(trc[:, 0], idt)])
                        and len(fr1) > 0)
            out["records_checked_videos"] = ids
            restore()
        dist.broadcast(ok, 0)
        out["records_equal_single_gpu_run"] = bool(int(ok.item()))
    # the reference arm's clip through the same API (rank 0, one video): the two arms on identical input
    if rank == 0:
        from articulation3d_b200 import workloads
        tr_, fr_ = REF_SAMPLE
        preds, _ = workloads.make_clip(wl, 2020, tracks=tr_, frames=fr_)      # the very clip the CPU port gets
        for p in preds:
            p.pred_masks = p.pred_masks.pin_memory()
        sv = [(p.pred_tran_axis.clone(), p.pred_rot_axis.clone(), p.pred_planes.clone()) for p in preds]
        best = None
        for _ in range(4):
            random.seed(2020)
            st = opt_utils.Stats()
            t0 = time.perf_counter()
            planes = opt_utils.track_planes(preds, cfg)
            opt_utils.optimize_planes(preds, planes, "3dc", cfg=cfg, device=dev, stats=st)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            for p, (ta, ra, pl) in zip(preds, sv):
                p.pred_tran_axis, p.pred_rot_axis, p.pred_planes = ta.clone(), ra.clone(), pl.clone()
            if best is None or dt < best[0]:
                best = (dt, st.units_visited)
        out["reference_sample"] = {"clip": f"{tr_} track x {fr_} frames of the {wl.name} clip shape, seed 2020 "
                                           f"(the clip `--impl reference` times)",
                                   "value": best[1] / best[0], "unit": UNIT, "ms": 1e3 * best[0], "units": best[1]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--e2e-videos", type=int, default=6, help="host clips per GPU of the e2e leg")
    ap.add_argument("--streams", type=int, default=1,
                    help="streams the timed steps alternate between; 2 was measured: 3 %% faster on a 256-job shard, "
                         "5 %% slower on the 2048-job headline (CTAs of two projection kernels interleave)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", dest="extras", action="store_false",
                    help="skip the extra single-video (c2) pass and the pack stream reported under 'extras'")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float32 / float64, at most "
                         f"{DUMP_BYTES // 10 ** 6} MB in all, seeded row samples of larger arrays): pass_* = the "
                         "device pass's PassResult, e2e_* = what the public API returned (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    from articulation3d_b200 import workloads
    wl = workloads.WORKLOADS[args.workload]
    if args.impl == "reference":
        reference_arm(args, wl)
    else:
        gpu_arm(args, wl)


if __name__ == "__main__":
    main()
