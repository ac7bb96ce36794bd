"""Cost of ``tools.opt_arti --override-depth`` at a realistic size.  Writes ``--videos`` clips of the configs[2]
shape (8 tracks x 120 frames at 640x480) carrying rendered depth (``synth.render_depths``), 147 MB of fp32 depth
per clip, so the default 17 clips hold 2.5 GB of depth, far more than the L2 cache.  In one process it reports:

* ``adapter.override_depth_records`` of all records loaded memory-mapped (as every rank loads them under
  torchrun): ms per clip, depth GB/s, peak device memory; twice, the second time with the file's pages cached.
* the parts it is made of, each over the same bytes: the host copy of the depth out of the mapped records into a
  pinned block, the pinned H2D copy of those bytes (as ``tools/h2d_probe.py``), and the device work (RLE decode and
  ``k_plane_offsets``, one ``override_depth_batch`` per clip with its depth already on the device);
* the per-record ``adapter.override_depth`` loop over ``--subset`` clips: its time and whether its planes equal
  the streamed ones;
* ``tools.opt_arti`` on the file with and without ``--override-depth``: its summary and override lines.

    python tools/override_depth_bench.py [--videos 17] [--subset 2] [--keep DIR]

Prints the card (``nvidia-smi --query-gpu=name,power.limit,clocks.max.sm``) first, then one JSON line per
measurement."""
from __future__ import annotations

import argparse
import contextlib
import io as _io
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from articulation3d_b200 import adapter, io, synth  # noqa: E402
from articulation3d_b200.tools import opt_arti  # noqa: E402

DEV = torch.device("cuda:0")


def emit(**kw):
    print(json.dumps(kw), flush=True)


def write_input(path, videos, seed):
    records = []
    for v in range(videos):
        preds, scene = synth.make_video(seed + v, 8, 120, device=DEV)
        records += io.preds_to_records(preds, video_id=f"synthetic{v:02d}_0_0", start_image_id=v * 10000,
                                       device=DEV, depths=synth.render_depths(scene, device=DEV))
    torch.save(records, path)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--videos", type=int, default=17)
    ap.add_argument("--subset", type=int, default=2, help="clips of the per-record override_depth loop")
    ap.add_argument("--seed", type=int, default=2020)
    ap.add_argument("--keep", default=None, help="keep the input and outputs in this directory")
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("override_depth_bench: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    emit(nvidia_smi=smi, torch=torch.__version__)

    work = args.keep or tempfile.mkdtemp(prefix="override_depth_bench_")
    os.makedirs(work, exist_ok=True)
    inp = os.path.join(work, "pred.pth")
    t0 = time.perf_counter()
    write_input(inp, args.videos, args.seed)
    torch.cuda.empty_cache()
    emit(input=f"{args.videos} clips x 8 tracks x 120 frames, 640x480, with pred_depth",
         file_bytes=os.path.getsize(inp), write_s=round(time.perf_counter() - t0, 1))

    # the streamed override, twice on fresh loads
    streamed = None
    for run in range(2):
        records = adapter.load_predictions(inp, mmap=True)
        nbytes = sum(r["pred_depth"].numel() * 4 for r in records if r["instances"])
        n_inst = sum(len(r["instances"]) for r in records)
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        dt, _ = timed(lambda: adapter.override_depth_records(records, DEV))
        emit(phase="override_depth_records", run=run, frames=len(records), instances=n_inst, depth_bytes=nbytes,
             ms=round(dt * 1e3, 1), ms_per_clip=round(dt * 1e3 / args.videos, 2),
             depth_gb_per_s=round(nbytes / dt / 1e9, 2),
             peak_device_mib=round((torch.cuda.max_memory_allocated() - base) / 2 ** 20, 1))
        streamed = [r["pred_plane"] for r in records]
        del records

    # its parts, over the same bytes
    records = adapter.load_predictions(inp, mmap=True)
    H, W = records[0]["pred_depth"].shape
    per_block = (256 << 20) // (H * W * 4)
    pinned = torch.empty(per_block, H, W, pin_memory=True)
    dev_block = torch.empty(per_block, H, W, device=DEV)

    def host_copy():
        for i, r in enumerate(records):
            pinned[i % per_block].copy_(r["pred_depth"])

    def h2d():
        for _ in range(-(-len(records) // per_block)):
            dev_block.copy_(pinned, non_blocking=True)
    for name, fn in (("host copy into pinned", host_copy), ("pinned H2D", h2d)):
        fn()
        ts = [timed(fn)[0] for _ in range(3)]
        emit(phase=name, bytes=len(records) * H * W * 4, ms_min=round(min(ts) * 1e3, 1),
             gb_per_s=round(len(records) * H * W * 4 / min(ts) / 1e9, 2))
    del pinned, dev_block
    groups = list(adapter.group_by_video(records).values())
    total = 0.0
    for k, recs in enumerate([groups[0]] + groups):           # the first clip once more as warm-up
        d = torch.stack([r["pred_depth"] for r in recs]).to(DEV)
        inst = [dict(instances=r["instances"], pred_plane=r["pred_plane"].clone()) for r in recs]
        dt, _ = timed(lambda: adapter.override_depth_batch(inst, depths=d))
        total += dt if k else 0.0
        del d
    emit(phase="device work (decode + plane_offsets, depth resident)", ms=round(total * 1e3, 1),
         ms_per_clip=round(total * 1e3 / len(groups), 2))

    # the per-record loop on a subset
    sub = [r for recs in groups[:args.subset] for r in recs]
    ref = streamed[:len(sub)]
    inst = [dict(instances=r["instances"], pred_plane=r["pred_plane"].clone()) for r in sub]

    def loop():
        return [adapter.override_depth(x, depth=r["pred_depth"].to(DEV)) for x, r in zip(inst, sub)]
    dt, out = timed(loop)
    equal = all(torch.equal(x["pred_plane"], p) for x, p in zip(out, ref))
    diff = max(float((x["pred_plane"] - p).abs().max()) for x, p in zip(out, ref) if p.numel())
    emit(phase="per-record override_depth loop", clips=args.subset, frames=len(sub), ms=round(dt * 1e3, 1),
         ms_per_clip=round(dt * 1e3 / args.subset, 2), planes_equal_streamed=equal, max_abs_diff=diff)
    del records, groups, sub, inst, out, streamed, ref
    torch.cuda.empty_cache()

    # the tool, with and without the flag
    for flag in ([], ["--override-depth"]):
        buf = _io.StringIO()
        out_dir = os.path.join(work, "out_override" if flag else "out_plain")
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(buf):
            opt_arti.main(["--input", inp, "--output", out_dir, "--seed", str(args.seed), "--device", "cuda:0",
                           *flag])
        emit(phase="tools.opt_arti", flags=flag, wall_s=round(time.perf_counter() - t0, 2),
             lines=buf.getvalue().splitlines())
        shutil.rmtree(out_dir, ignore_errors=True)
    if not args.keep:
        shutil.rmtree(work, ignore_errors=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
