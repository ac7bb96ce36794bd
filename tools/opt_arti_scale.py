"""Scaling of ``tools.opt_arti`` over the GPUs of one box.  Writes one synthetic ``.pth`` of the configs[2] clip
shape (``--videos`` clips of 8 tracks x 120 frames at 640x480, masks encoded on cuda:0), then runs the tool on it
under ``python -m torch.distributed.run --standalone --nnodes 1 --nproc-per-node N`` for every N of 1, 2, 4, 8 the
box has, each N into its own output directory:

    python tools/opt_arti_scale.py [--videos 64] [--gpus 1,2,4,8] [--timeout 1800] [--keep DIR]

Prints the card (``nvidia-smi --query-gpu=name,power.limit,clocks.max.sm``), then one JSON line per N: videos,
evaluations, the tool's optimise time (its summary line: the slowest rank), evaluations/s and its ratio to N x
the N = 1 figure, the tool's wall time per rank from the start of ``main`` (load, conversion, tracking, optimise,
writes; interpreter and torch start-up excluded) with the host time of its phases outside the optimisation, the
launch's wall time, peak RSS per rank, and whether every output file equals the N = 1 run's.  Peak RSS counts
every resident page of the memory-mapped input in every rank, so it does not show the sharing of those pages;
the proportional set size (PSS, /proc/self/smaps_rollup) at the tool's return divides shared pages among the
processes that map them.  Every rank runs with OMP_NUM_THREADS=1
(INTEGRATION.md §1).  Exits non-zero if a run fails or an output differs."""
from __future__ import annotations

import argparse
import json
import os
import re
import resource
import signal
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

SUMMARY = re.compile(r"^(\d+) video\(s\), (\d+) track\(s\): (\d+) track-frame x candidate evaluations in ([0-9.]+) ms "
                     r"\((\d+) device passes\)")
WORKER = "--rank-worker"


def rank_worker(stats_dir, tool_args):
    """One torchrun rank: the tool's ``main``, then its wall time, the host time of its phases outside the
    optimisation, its peak RSS and its PSS at the return to ``stats_dir/rank<r>.json``."""
    from articulation3d_b200 import adapter, io, opt_utils
    from articulation3d_b200.tools import opt_arti
    phases = {}

    def timed(mod, name, phase):
        fn = getattr(mod, name)

        def wrapper(*a, **k):
            t = time.perf_counter()
            try:
                return fn(*a, **k)
            finally:
                phases[phase] = phases.get(phase, 0.0) + time.perf_counter() - t
        setattr(mod, name, wrapper)
    for mod, name, phase in ((adapter, "load_predictions", "load"), (adapter, "group_by_video", "group"),
                             (opt_arti, "frame_config", "group"), (io, "records_to_preds", "convert"),
                             (opt_utils, "track_planes", "track"), (io, "save_results", "write"),
                             (io, "write_obj", "write")):
        timed(mod, name, phase)
    t0 = time.perf_counter()
    opt_arti.main(tool_args)
    wall = time.perf_counter() - t0
    rss_mib = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1024      # KiB on Linux
    with open("/proc/self/smaps_rollup") as f:                                # kB
        pss_mib = next(int(l.split()[1]) for l in f if l.startswith("Pss:")) / 1024
    with open(os.path.join(stats_dir, f"rank{os.environ.get('RANK', '0')}.json"), "w") as f:
        json.dump({"wall_s": wall, "phases_s": phases, "peak_rss_mib": rss_mib, "pss_mib_at_exit": pss_mib}, f)


def _descendants(pid):
    children = {}
    for d in os.listdir("/proc"):
        try:
            with open(f"/proc/{d}/stat") as f:
                children.setdefault(int(f.read().rsplit(")", 1)[1].split()[1]), []).append(int(d))
        except (OSError, ValueError, IndexError):
            continue
    out, todo = [], [pid]
    while todo:
        for c in children.get(todo.pop(), []):
            out.append(c)
            todo.append(c)
    return out


def run(cmd, timeout, env):
    """``cmd`` -> (return code, stdout, stderr).  torchrun starts every worker in a session of its own, so on a
    timeout the whole process tree is killed, not just the launcher, and the timeout is re-raised."""
    proc = subprocess.Popen(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                            start_new_session=True)
    try:
        out, err = proc.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        for p in _descendants(proc.pid) + [proc.pid]:
            try:
                os.kill(p, signal.SIGKILL)
            except ProcessLookupError:
                pass
        proc.communicate()
        raise
    return proc.returncode, out, err


def same(a, b) -> bool:
    if isinstance(a, torch.Tensor):
        return isinstance(b, torch.Tensor) and a.dtype == b.dtype and torch.equal(a, b)
    if isinstance(a, dict):
        return isinstance(b, dict) and a.keys() == b.keys() and all(same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return type(a) is type(b) and len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    return type(a) is type(b) and bool(a == b)


def same_outputs(want_dir, got_dir) -> bool:
    """Same file names; ``.pth`` records equal after loading, every other file equal byte for byte."""
    files = sorted(os.listdir(want_dir))
    if files != sorted(os.listdir(got_dir)):
        return False
    for name in files:
        a, b = os.path.join(want_dir, name), os.path.join(got_dir, name)
        if name.endswith(".pth"):
            if not same(torch.load(a, weights_only=False), torch.load(b, weights_only=False)):
                return False
        else:
            with open(a, "rb") as fa, open(b, "rb") as fb:
                if fa.read() != fb.read():
                    return False
    return True


def write_input(path, videos, seed):
    from articulation3d_b200 import io, synth
    records = []
    for v in range(videos):
        preds, _ = synth.make_video(seed + v, 8, 120, device="cuda:0")
        records += io.preds_to_records(preds, video_id=f"synthetic{v:02d}_0_0", start_image_id=v * 10000,
                                       device="cuda:0")
    torch.save(records, path)


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--videos", type=int, default=64)
    ap.add_argument("--seed", type=int, default=2020)
    ap.add_argument("--gpus", default="1,2,4,8", help="world sizes to run (those above the box's GPU count are "
                    "skipped); the first is the reference for the ratios and the output check")
    ap.add_argument("--timeout", type=float, default=1800, help="seconds per torchrun launch")
    ap.add_argument("--keep", default=None, help="keep the input and outputs in this directory")
    args = ap.parse_args(argv)
    n_dev = torch.cuda.device_count()
    if n_dev == 0:
        raise SystemExit("opt_arti_scale: no CUDA device")
    sizes = [n for n in map(int, args.gpus.split(",")) if n <= n_dev]
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    print(json.dumps({"gpus_on_box": n_dev, "nvidia_smi": smi}), flush=True)

    work = args.keep or tempfile.mkdtemp(prefix="opt_arti_scale_")
    os.makedirs(work, exist_ok=True)
    inp = os.path.join(work, "pred.pth")
    t0 = time.perf_counter()
    write_input(inp, args.videos, args.seed)
    torch.cuda.empty_cache()
    print(json.dumps({"input": f"{args.videos} videos x 8 tracks x 120 frames, 640x480", "bytes":
                      os.path.getsize(inp), "write_s": round(time.perf_counter() - t0, 1)}), flush=True)

    env = dict(os.environ, OMP_NUM_THREADS="1")
    env["PYTHONPATH"] = os.pathsep.join(p for p in (ROOT, env.get("PYTHONPATH")) if p)
    ok, ref = True, None
    for n in sizes:
        out_dir, stats_dir = os.path.join(work, f"out_n{n}"), os.path.join(work, f"stats_n{n}")
        os.makedirs(stats_dir, exist_ok=True)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nnodes", "1", "--nproc-per-node",
               str(n), os.path.abspath(__file__), WORKER, stats_dir,
               "--input", inp, "--output", out_dir, "--seed", str(args.seed)]
        t0 = time.perf_counter()
        rc, out, err = run(cmd, args.timeout, env)
        launch_s = time.perf_counter() - t0
        m = [SUMMARY.match(l) for l in out.splitlines() if SUMMARY.match(l)]
        if rc != 0 or len(m) != 1:
            print(json.dumps({"n_gpus": n, "returncode": rc, "stderr_tail": err[-3000:]}), flush=True)
            ok = False
            continue
        videos, tracks, units, opt_ms, passes = (float(x) if i == 3 else int(x) for i, x in enumerate(m[0].groups()))
        ranks = [json.load(open(os.path.join(stats_dir, f"rank{r}.json"))) for r in range(n)]
        rate = units / (opt_ms / 1e3)
        if ref is None:
            ref = (n, rate, out_dir)
        equal = same_outputs(ref[2], out_dir)
        ok &= equal
        print(json.dumps({
            "n_gpus": n, "videos": videos, "tracks": tracks, "evaluations": units, "device_passes": passes,
            "optimise_ms_max_over_ranks": opt_ms, "evaluations_per_s": round(rate),
            f"ratio_to_n_x_n{ref[0]}": round(rate / (n / ref[0] * ref[1]), 3),
            "tool_wall_s_per_rank": [round(r["wall_s"], 2) for r in ranks],
            "host_phases_s_per_rank": [{k: round(v, 2) for k, v in r["phases_s"].items()} for r in ranks],
            "launch_wall_s": round(launch_s, 1),
            "peak_rss_mib_per_rank": [round(r["peak_rss_mib"]) for r in ranks],
            "pss_mib_at_exit_per_rank": [round(r["pss_mib_at_exit"]) for r in ranks],
            "outputs_equal_first_run": equal}), flush=True)
    if not args.keep:
        import shutil
        shutil.rmtree(work, ignore_errors=True)
    if not ok:
        print("opt_arti_scale: a run failed or its outputs differ from the first run's", file=sys.stderr)
        return 1
    return 0


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == WORKER:
        rank_worker(sys.argv[2], sys.argv[3:])
    else:
        sys.exit(main())
