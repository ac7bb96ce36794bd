"""Cost of writing masks as COCO RLE, host encoder against the GPU encoder, on a configs[2]-shaped clip
(8 tracks x 120 frames, 640x480, synth.make_video(2020, 8, 120)):

  (a) io.preds_to_records on the host path and with device="cuda:0" (records must be equal);
  (b) per fitted track of the optimised clip, RegMasks.to_rle() against reg_masks[f] + rle.encode per frame
      (the two must give equal bytes);
  (c) the two kernels alone on the clip's 960 packed masks: CUDA events over many launches with L2 overwritten
      between launches, and the engine call's D2H copy and the host string writer timed separately.

    python tools/rle_bench.py [--reps 5] [--launches 200]

Prints the card's name and power limit, then one JSON line per measurement.  Exits non-zero if a check fails."""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from articulation3d_b200 import _lib, engine, io, opt_utils, rle, synth  # noqa: E402

DEV = "cuda:0"


def card() -> dict:
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except (OSError, ValueError, subprocess.SubprocessError):
        out["power_limit"] = "unknown"
    return out


def wall(fn, reps):
    """Median wall time (ms) of fn(), each run ending in a device synchronise."""
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), r


def emit(**kw):
    print(json.dumps(kw), flush=True)


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--launches", type=int, default=200)
    args = ap.parse_args(argv)
    torch.zeros(1, device=DEV)
    _lib.load()
    emit(**card())
    ok = True
    preds, _ = synth.make_video(2020, 8, 120)
    n_masks = sum(len(p.pred_masks) for p in preds)
    H, W = preds[0].pred_masks.shape[1:]

    # (a) the records writer
    io.preds_to_records(preds[:2], device=DEV)                       # module load, allocator
    t_host, rec_h = wall(lambda: io.preds_to_records(preds), max(1, args.reps // 2))
    t_dev, rec_d = wall(lambda: io.preds_to_records(preds, device=DEV), args.reps)
    same = [r["instances"] for r in rec_h] == [r["instances"] for r in rec_d]
    ok &= same
    emit(what="a_preds_to_records", masks=n_masks, host_ms=round(t_host, 2), device_ms=round(t_dev, 2),
         host_ms_per_mask=round(t_host / n_masks, 4), device_ms_per_mask=round(t_dev / n_masks, 4), equal=same)

    # (b) registered masks of the optimised clip
    random.seed(2020)
    planes = opt_utils.track_planes(preds)
    t_opt, _ = wall(lambda: opt_utils.optimize_planes(preds, planes, '3dc', device=DEV), 1)
    fitted = [p for c in ("trans", "rot") for p in planes[c] if p.get("has_rot")]
    t_gpu = t_cpu = 0.0
    frames = 0
    same = True
    for p in fitted:
        rm = p["reg_masks"]
        dt, got = wall(rm.to_rle, args.reps)
        t_gpu += dt

        def per_frame():
            fresh = opt_utils.RegMasks(list(rm), rm.packed, H, W)       # no cached images
            return {f: rle.encode(np.asarray(fresh[f])) for f in fresh}
        dt, want = wall(per_frame, 1)
        t_cpu += dt
        frames += len(rm)
        same &= got == want
    ok &= same
    emit(what="b_reg_masks", tracks=len(fitted), frames=frames, optimize_ms=round(t_opt, 2),
         to_rle_ms=round(t_gpu, 2), per_frame_emit_encode_ms=round(t_cpu, 2),
         d2h_bytes_per_frame_path=frames * H * W * 4, equal=same)

    # (c) the kernels alone on the clip's packed masks
    lib = _lib.load()
    pb = engine.PoolBuilder(n_masks, H, W, DEV)
    for p in preds:
        pb.append(p.pred_masks.to(DEV))
    bits = pb.bits
    s = torch.cuda.current_stream().cuda_stream
    runs = torch.empty(n_masks, dtype=torch.int64, device=DEV)
    begin = torch.zeros(n_masks + 1, dtype=torch.int64, device=DEV)
    lib.a3d_rle_count_runs(bits.data_ptr(), None, n_masks, H, W, runs.data_ptr(), s)
    begin[1:] = torch.cumsum(runs, 0)
    total = int(begin[-1])
    counts = torch.empty(total, dtype=torch.int32, device=DEV)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)    # twice the 126 MB of L2
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.launches)]
    kernel_ms = {}
    for name, launch in (("k_rle_count", lambda: lib.a3d_rle_count_runs(bits.data_ptr(), None, n_masks, H, W,
                                                                          runs.data_ptr(), s)),
                         ("k_bits_to_rle", lambda: lib.a3d_bits_to_rle(bits.data_ptr(), None, n_masks, H, W,
                                                                       begin.data_ptr(), counts.data_ptr(), s))):
        for _ in range(5):
            _lib.check(launch(), name)
        for a, b in ev:
            flush.fill_(1)
            a.record()
            launch()
            b.record()
        torch.cuda.synchronize()
        kernel_ms[name] = float(np.median([a.elapsed_time(b) for a, b in ev]))
    packed_bytes = bits.numel() * 4
    ref_counts, ref_begin = engine.bits_to_rle(bits, H, W)
    same = np.array_equal(counts.cpu().numpy().view(np.uint32), ref_counts) and \
        np.array_equal(begin.cpu().numpy(), ref_begin)
    ok &= same
    t_call, (fc, fb) = wall(lambda: engine.bits_to_rle(bits, H, W), args.reps)
    block = torch.empty(n_masks + 1 + (total + 1) // 2, dtype=torch.int64, device=DEV)
    t_d2h, _ = wall(lambda: block.cpu(), args.reps)
    t_str, strings = wall(lambda: rle.counts_to_strings(fc, fb), args.reps)
    emit(what="c_kernels", masks=n_masks, shape=[H, W], runs=total, packed_bytes=packed_bytes,
         k_rle_count_us=round(kernel_ms["k_rle_count"] * 1e3, 2),
         k_bits_to_rle_us=round(kernel_ms["k_bits_to_rle"] * 1e3, 2),
         k_rle_count_GBps=round(packed_bytes / kernel_ms["k_rle_count"] / 1e6, 1),
         k_bits_to_rle_GBps=round(packed_bytes / kernel_ms["k_bits_to_rle"] / 1e6, 1),
         engine_call_ms=round(t_call, 3), d2h_ms=round(t_d2h, 3), d2h_bytes=block.numel() * 8,
         host_strings_ms=round(t_str, 3), string_bytes=sum(len(x) for x in strings), l2="overwritten between launches",
         equal=bool(same))
    if not ok:
        print("rle_bench: an equality check failed", file=sys.stderr)
        return 1
    return 0


if __name__ == "__main__":
    sys.exit(main())
