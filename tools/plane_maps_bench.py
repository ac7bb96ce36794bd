"""Cost of the fitted planes' depth and normal maps (render.plane_maps / a3d_plane_maps) on two clips: a
configs[2]-shaped one (8 tracks x 120 frames, 640x480, synth.make_video(2020, 8, 120)) and a 300-frame one
(4 tracks x 300 frames, 640x480), both optimised with optimize_planes('3dc') first:

  (a) k_plane_maps alone, lists and pool resident: median of CUDA events per launch with L2 overwritten between
      launches; GB/s of the algorithmic bytes (4 + 3 bytes written per pixel, + the packed words inside every
      layer's box) and their share of the HBM rate a device copy reaches in the same run; the float64 operations
      of the (pixel, covering layer) pairs (ray 4, dot 5, division 1, z 1 for the sparse intrinsics) per second;
      the first frames are checked bit for bit against tests/plane_maps_ref.py;
  (b) render.plane_maps whole (layer lists, pool, upload, kernel);
  (c) the host side of render.write_plane_maps: PNG + mp4 encoding of the maps alone, and write_plane_maps whole.

    python tools/plane_maps_bench.py [--launches 50]

Prints the card's name, power limit and max SM clock, then one JSON line per measurement.  Exits non-zero if a
check fails."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from articulation3d_b200 import OptConfig, _lib, engine, render  # noqa: E402
from tests import plane_maps_ref  # noqa: E402
from tools.render_bench import card, clip, emit, hbm_copy_gbs, median_event_ms  # noqa: E402  (same clips, same timing)

DEV = "cuda:0"
CHECK_FRAMES = 6
F64_OPS_SPARSE = 4 + 5 + 1 + 1         # rx, ry (2 + 2); dot (3 products, 2 sums); division; depth * rz


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
    lib = _lib.load()
    for name, seed, tracks, frames in (("configs2_8x120", 2020, 8, 120), ("clip_4x300", 2021, 4, 300)):
        opt, planes = clip(seed, tracks, frames, cfg)
        T = len(opt)
        lists = render.plane_lists(opt, planes, cfg)
        pool = render.mask_pool(opt, lists, cfg, torch.device(DEV))
        d_lay = torch.from_numpy(np.ascontiguousarray(lists.layers).view(np.uint8).copy()).to(DEV)
        d_lb = torch.from_numpy(lists.layer_begin).to(DEV)
        depth = torch.empty(T, H, W, dtype=torch.float32, device=DEV)
        rgb = torch.empty(T, H, W, 3, dtype=torch.uint8, device=DEV)
        cam = engine.camera_struct(cfg)
        bg = (ctypes.c_uint8 * 3)(0, 0, 0)
        stream = torch.cuda.current_stream().cuda_stream

        def launch():
            _lib.check(lib.a3d_plane_maps(ctypes.byref(cam), T, pool.bits.data_ptr(), pool.bbox.data_ptr(), len(pool),
                                          d_lay.data_ptr(), d_lb.data_ptr(), bg, depth.data_ptr(), rgb.data_ptr(),
                                          stream), "a3d_plane_maps")
        launch()
        torch.cuda.synchronize()
        # check: the first frames bit for bit against the restatement
        lb = lists.layer_begin
        sub = lists.layers[:lb[CHECK_FRAMES]].copy()
        used, sub["mask"] = np.unique(sub["mask"], return_inverse=True)          # only the masks those frames draw
        masks = engine.emit_masks(pool.bits, torch.from_numpy(used.astype(np.int32)).to(DEV), H, W,
                                  dtype=torch.uint8).cpu().numpy()
        want_d, want_c = plane_maps_ref.plane_maps(cfg.K_inv(), masks, sub, lb[:CHECK_FRAMES + 1])
        equal = bool(np.array_equal(depth[:CHECK_FRAMES].cpu().numpy().view(np.int32), want_d.view(np.int32))
                     and np.array_equal(rgb[:CHECK_FRAMES].cpu().numpy(), want_c))
        ok &= equal
        ms = median_event_ms(launch, args.launches, flush)
        bb = pool.bbox.cpu().numpy().astype(np.int64)[lists.layers["mask"]]
        mask_bytes = int((np.maximum(bb[:, 1] - bb[:, 0] + 1, 0) * np.maximum(bb[:, 3] - bb[:, 2] + 1, 0) * 4).sum())
        nbytes = T * H * W * (4 + 3) + mask_bytes
        pairs = int(pool.popc.cpu().numpy().astype(np.int64)[lists.layers["mask"]].sum())
        emit(what="k_plane_maps", clip=name, frames=T, layers=len(lists.layers), covered_pairs=pairs,
             us=round(ms * 1e3, 1), algorithmic_bytes=nbytes, gbs=round(nbytes / ms / 1e6, 1),
             share_of_copy_rate=round(nbytes / ms / 1e6 / peak, 3), f64_ops=pairs * F64_OPS_SPARSE,
             f64_gflops=round(pairs * F64_OPS_SPARSE / ms / 1e6, 1), l2="overwritten between launches",
             first_frames_bit_equal_to_restatement=equal)
        # (b) plane_maps whole
        times = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            render.plane_maps(opt, planes, cfg=cfg, device=DEV)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        emit(what="plane_maps", clip=name, frames=T, ms=round(float(np.median(times)) * 1e3, 2))
        # (c) host encode of the maps alone, and write_plane_maps whole
        mm = render.depth_millimetres(depth).cpu().numpy().view(np.uint16)
        host_rgb = rgb.cpu().numpy()
        with tempfile.TemporaryDirectory() as tmp:
            t0 = time.perf_counter()
            for k, d in enumerate(mm):
                cv2.imwrite(os.path.join(tmp, f"{k:05d}.png"), d)
            t_png = time.perf_counter() - t0
            writer = cv2.VideoWriter(os.path.join(tmp, "a.mp4"), cv2.VideoWriter_fourcc(*"mp4v"), 30.0, (W, H))
            t0 = time.perf_counter()
            for fr in host_rgb:
                writer.write(cv2.cvtColor(fr, cv2.COLOR_RGB2BGR))
            writer.release()
            t_enc = time.perf_counter() - t0
            t0 = time.perf_counter()
            render.write_plane_maps(tmp, "b", opt, planes, cfg=cfg, device=DEV)
            t_w = time.perf_counter() - t0
        emit(what="encode", clip=name, frames=T, png_ms=round(t_png * 1e3, 1), cv2_mp4v_ms=round(t_enc * 1e3, 1),
             write_plane_maps_ms=round(t_w * 1e3, 1))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
