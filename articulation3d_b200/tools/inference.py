"""Temporal stage of the reference's ``tools/inference.py`` (:249-250) on a clip of
detections.  The R-CNN itself is out of scope (it stays in the reference's detectron2
code); without it this tool runs on the synthetic detector stub (``synth.make_video``),
which emits the same ``Instances`` contract:

    python -m articulation3d_b200.tools.inference --frames 30 --tracks 4 --output out/ [--save-obj] [--save-textured-obj] \
        [--save-masks] [--save-video [--fps 30]] [--save-depth]

``--save-obj`` writes the geometry-only quads of ``io.write_obj``; ``--save-textured-obj`` the reference's export
(``save_obj_model``, tools/inference.py:44-168, :282: object, rotated copies, axis markers, background, one
300x300 texture each) through ``articulation3d_b200.export`` — with a flat grey image, the stub has no video.
``--save-masks`` adds every fitted frame's registered mask to ``<id>_tracks.json`` as COCO RLE (``segmentation`` of
each ``angle_track`` entry).  ``--save-video`` writes ``<id>.mp4``: every frame drawn with the fitted result
(``render.write_video``: registered masks, detection outlines, axes; reference tools/inference.py:253-278) on a flat
grey background.  ``--save-depth`` writes the fitted planes' per-frame depth as ``<id>_depth/<k:05d>.png`` (uint16
millimetres, 0 = no plane) and their surface normals as ``<id>_normals.mp4`` (``render.write_plane_maps``; reference
tools/inference.py:231-243 shows the normal map).
"""
from __future__ import annotations

import argparse
import os
import random
import time

import torch

from articulation3d_b200 import OptConfig, io, opt_utils, synth


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--output", required=True)
    ap.add_argument("--frames", type=int, default=30)
    ap.add_argument("--tracks", type=int, default=4)
    ap.add_argument("--seed", type=int, default=2020)
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--save-obj", action="store_true")
    ap.add_argument("--save-textured-obj", action="store_true")
    ap.add_argument("--save-masks", action="store_true", help="registered masks (COCO RLE) in the tracks JSON")
    ap.add_argument("--save-video", action="store_true", help="<output>/synthetic00_0_0.mp4 of the fitted result")
    ap.add_argument("--fps", type=float, default=30)
    ap.add_argument("--save-depth", action="store_true", help="<output>/synthetic00_0_0_depth/<k>.png (uint16 mm) and "
                    "synthetic00_0_0_normals.mp4 of the fitted planes")
    args = ap.parse_args(argv)
    random.seed(args.seed)                                   # tools/inference.py:172
    cfg = OptConfig()
    preds, _ = synth.make_video(args.seed, args.tracks, args.frames, cfg)
    records = io.preds_to_records(preds, video_id="synthetic00_0_0", device=args.device)
    torch.zeros(1, device=args.device)                       # CUDA context and library load are not the optimiser's time
    opt_utils._lib.load()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    planes = opt_utils.track_planes(preds, cfg)
    opt_preds = opt_utils.optimize_planes(preds, planes, '3dc', cfg=cfg, device=args.device)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    io.save_results(args.output, "synthetic00_0_0", io.opt_preds_to_records(opt_preds, records), planes,
                    masks=args.save_masks)
    if args.save_obj:
        for k in sorted({0, min(30, args.frames - 1), min(60, args.frames - 1), min(89, args.frames - 1)}):
            io.write_obj(os.path.join(args.output, f"frame{k}.obj"), opt_preds, planes, k, cfg)   # inference.py:282
    if args.save_textured_obj:
        from articulation3d_b200 import export
        for k in sorted({0, min(30, args.frames - 1), min(60, args.frames - 1), min(89, args.frames - 1)}):
            export.save_obj_model(args.output, opt_preds, k, image=None, cfg=cfg)                 # inference.py:282
    if args.save_video:
        from articulation3d_b200 import render
        render.write_video(os.path.join(args.output, "synthetic00_0_0.mp4"), opt_preds, planes, fps=args.fps,
                           cfg=cfg, device=args.device)
    if args.save_depth:
        from articulation3d_b200 import render
        render.write_plane_maps(args.output, "synthetic00_0_0", opt_preds, planes, fps=args.fps, cfg=cfg,
                                device=args.device)
    print(f"{args.frames} frames, {len(planes['rot'])} rot + {len(planes['trans'])} trans tracks "
          f"in {dt * 1e3:.1f} ms -> {args.output}")


if __name__ == "__main__":
    main()
