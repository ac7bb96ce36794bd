"""Cost of drawing the fitted result into the clip's frames (render.render_clip / a3d_render) on two clips:
a configs[2]-shaped one (8 tracks x 120 frames, 640x480, synth.make_video(2020, 8, 120)) and a 300-frame one
(4 tracks x 300 frames, 640x480):

  (a) a3d_render alone, lists and pool resident: CUDA events per launch with L2 overwritten between launches;
      GB/s of the algorithmic bytes (3 H W written per frame, + 3 H W read per frame with a per-frame
      background, + the packed words inside every drawn layer's box) and their share of the HBM rate a device
      copy reaches in the same run (grey shared background, and per-frame random backgrounds);
  (b) render.render_clip whole (draw lists, pool, upload, kernel), and the D2H copy of its frames to pinned memory;
  (c) the host alternative: reg_masks[f] dense per frame plus numpy compositing of the same lists
      (tests/render_ref.py), which must equal (b) byte for byte;
  (d) cv2 mp4v encoding of the frames (RGB -> BGR, VideoWriter.write), and render.write_video whole.

    python tools/render_bench.py [--launches 50]

Prints the card's name and power limit, then one JSON line per measurement.  Exits non-zero if a check fails."""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from articulation3d_b200 import OptConfig, _lib, opt_utils, render, synth  # noqa: E402
from articulation3d_b200.opt_utils import RegMasks  # noqa: E402
from tests import render_ref  # noqa: E402

DEV = "cuda:0"


def card() -> dict:
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception:
        out["power_limit"] = "unknown"
    return out


def emit(**kw):
    print(json.dumps(kw), flush=True)


def median_event_ms(fn, launches: int, flush: torch.Tensor) -> float:
    times = []
    for _ in range(launches):
        flush.fill_(1)                                  # L2 overwritten between launches
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times))


def hbm_copy_gbs(flush: torch.Tensor) -> float:
    src = torch.empty(1 << 30, dtype=torch.uint8, device=DEV)
    dst = torch.empty_like(src)
    dst.copy_(src)
    ms = median_event_ms(lambda: dst.copy_(src), 10, flush)
    return 2 * src.numel() / ms / 1e6


def clip(seed: int, tracks: int, frames: int, cfg: OptConfig):
    preds, _ = synth.make_video(seed, tracks, frames, cfg)
    random.seed(seed)
    planes = opt_utils.track_planes(preds, cfg)
    out = opt_utils.optimize_planes(preds, planes, '3dc', cfg=cfg, device=DEV)
    torch.cuda.synchronize()
    return out, planes


def layer_bytes(pool, lists) -> int:
    """Packed words inside the box of every drawn layer (what the kernel reads of the pool)."""
    bb = pool.bbox.cpu().numpy().astype(np.int64)[lists.layers["mask"]]
    return int((np.maximum(bb[:, 1] - bb[:, 0] + 1, 0) * np.maximum(bb[:, 3] - bb[:, 2] + 1, 0) * 4).sum())


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--launches", type=int, default=50)
    args = ap.parse_args(argv)
    import cv2
    torch.cuda.set_device(0)
    info = card()
    print(f"# {info}", flush=True)
    cfg = OptConfig()
    H, W = cfg.height, cfg.width
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)      # twice the 126 MB of L2
    peak = hbm_copy_gbs(flush)
    emit(what="hbm_copy", gbs=round(peak, 1), note="device-to-device copy of 1 GiB, read + write bytes", **info)
    ok = True
    for name, seed, tracks, frames in (("configs2_8x120", 2020, 8, 120), ("clip_4x300", 2021, 4, 300)):
        opt, planes = clip(seed, tracks, frames, cfg)
        T = len(opt)
        lists = render.draw_lists(opt, planes, cfg)
        pool = render.mask_pool(opt, lists, cfg, torch.device(DEV))
        lib = _lib.load()
        dev = [torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).copy()).to(DEV)
               for a in (lists.layers, lists.layer_begin, lists.segs, lists.seg_begin)]
        out = torch.empty(T, H, W, 3, dtype=torch.uint8, device=DEV)
        grey = torch.full((H, W, 3), 160, dtype=torch.uint8, device=DEV)
        frames_bg = torch.randint(0, 256, (T, H, W, 3), dtype=torch.uint8, device=DEV)
        lbytes = layer_bytes(pool, lists)
        stream = torch.cuda.current_stream().cuda_stream
        for bg_name, bg, stride in (("shared", grey, 0), ("per_frame", frames_bg, H * W * 3)):
            def launch():
                _lib.check(lib.a3d_render(bg.data_ptr(), stride, T, H, W, pool.bits.data_ptr(), pool.bbox.data_ptr(),
                                          len(pool), dev[0].data_ptr(), dev[1].data_ptr(), dev[2].data_ptr(),
                                          dev[3].data_ptr(), out.data_ptr(), stream), "a3d_render")
            launch()
            ms = median_event_ms(launch, args.launches, flush)
            nbytes = T * H * W * 3 * (2 if stride else 1) + lbytes
            emit(what="a3d_render", clip=name, frames=T, background=bg_name, layers=len(lists.layers),
                 segments=len(lists.segs), us=round(ms * 1e3, 1), algorithmic_bytes=nbytes,
                 gbs=round(nbytes / ms / 1e6, 1), share_of_copy_rate=round(nbytes / ms / 1e6 / peak, 3),
                 l2="overwritten between launches")
        # (b) render_clip whole, then its D2H
        times = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            frames_dev = render.render_clip(opt, planes, cfg=cfg, device=DEV)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        host = torch.empty(frames_dev.shape, dtype=torch.uint8).pin_memory()
        d2h = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            host.copy_(frames_dev, non_blocking=True)
            torch.cuda.synchronize()
            d2h.append(time.perf_counter() - t0)
        emit(what="render_clip", clip=name, frames=T, ms=round(float(np.median(times)) * 1e3, 2),
             d2h_ms=round(float(np.median(d2h)) * 1e3, 2), d2h_bytes=host.numel(),
             d2h_gbs=round(host.numel() / float(np.median(d2h)) / 1e9, 1))
        # (c) host alternative: dense registered masks (fresh RegMasks: nothing cached) + numpy compositing
        t0 = time.perf_counter()
        masks = []
        for pl in lists.fitted:
            rm = RegMasks(list(pl["ids"].keys()), pl["reg_masks"].packed, H, W)
            masks += [rm[f].numpy() > 0.5 for f in pl["ids"]]
        t_dense = time.perf_counter() - t0
        det = [m.numpy() > 0.5 for p in opt for m in p.pred_masks]
        t0 = time.perf_counter()
        want = render_ref.composite(np.full((H, W, 3), 160, np.uint8), np.stack(masks + det), lists.layers,
                                    lists.layer_begin, lists.segs, lists.seg_begin)
        t_comp = time.perf_counter() - t0
        equal = bool(np.array_equal(host.numpy(), want))
        ok &= equal
        emit(what="host_alternative", clip=name, frames=T, reg_masks_dense_ms=round(t_dense * 1e3, 1),
             numpy_composite_ms=round(t_comp * 1e3, 1), byte_equal_to_render_clip=equal)
        # (d) cv2 encode of the frames, and write_video whole
        with tempfile.TemporaryDirectory() as tmp:
            writer = cv2.VideoWriter(os.path.join(tmp, "a.mp4"), cv2.VideoWriter_fourcc(*"mp4v"), 30.0, (W, H))
            t0 = time.perf_counter()
            for fr in host.numpy():
                writer.write(cv2.cvtColor(fr, cv2.COLOR_RGB2BGR))
            writer.release()
            t_enc = time.perf_counter() - t0
            t0 = time.perf_counter()
            render.write_video(os.path.join(tmp, "b.mp4"), opt, planes, cfg=cfg, device=DEV)
            t_wv = time.perf_counter() - t0
        emit(what="encode", clip=name, frames=T, cv2_mp4v_ms=round(t_enc * 1e3, 1), write_video_ms=round(t_wv * 1e3, 1))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
