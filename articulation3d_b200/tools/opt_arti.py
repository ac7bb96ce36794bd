"""Temporal optimisation of saved predictions — the B200 counterpart of the reference's
``tools/opt_arti.py`` for the stage in scope (the detector is not re-run):

    python -m articulation3d_b200.tools.opt_arti --input instances_predictions.pth --output out/ [--save-obj] [--save-masks]

Reads the per-frame prediction records (RLE masks stay run-length encoded and are decoded on
the GPU), groups them by video, runs ``track_planes`` + ``optimize_planes('3dc')`` for all videos
in lock-step, and writes per video ``<id>_predictions_opt.pth`` (records as
tools/opt_arti.py:229-249), ``<id>_tracks.json`` (fitted axis + angle-per-frame track) and
optionally ``<id>_frame<k>.obj``; ``--save-masks`` adds every fitted frame's registered mask to the tracks JSON
as COCO RLE.  ``--synthetic N`` writes a synthetic input first (masks encoded on ``--device``).
"""
from __future__ import annotations

import argparse
import os
import time

import torch

from articulation3d_b200 import OptConfig, adapter, io, opt_utils, synth


def frame_index(record) -> int:
    """Trailing integer of the file name (``<yt id>_<shot>_<frame>_<offset>.png``)."""
    stem = os.path.splitext(os.path.basename(record["file_name"]))[0]
    return int(stem.split("_")[-1])


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--input", required=True)
    ap.add_argument("--output", required=True)
    ap.add_argument("--conf-threshold", type=float, default=0.7)
    ap.add_argument("--seed", type=int, default=2020, help="per-video RNG seed base (tools/inference.py:172)")
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--save-obj", action="store_true")
    ap.add_argument("--save-masks", action="store_true", help="registered masks (COCO RLE) in the tracks JSON")
    ap.add_argument("--gt-json", default=None, help="COCO-style ground truth: print the AP table before / after "
                    "optimisation (tools/opt_arti.py:275-283)")
    ap.add_argument("--synthetic", type=int, default=0, help="first write N synthetic videos to --input")
    ap.add_argument("--tracks", type=int, default=4)
    ap.add_argument("--frames", type=int, default=60)
    args = ap.parse_args(argv)

    if args.synthetic:
        records = []
        for v in range(args.synthetic):
            preds, _ = synth.make_video(args.seed + v, args.tracks, args.frames)
            records += io.preds_to_records(preds, video_id=f"synthetic{v:02d}_0_0", start_image_id=v * 10000,
                                           device=args.device)
        torch.save(records, args.input)

    cfg = OptConfig()
    groups = adapter.group_by_video(adapter.load_predictions(args.input))
    videos, order = [], []
    for vid, recs in groups.items():
        preds = io.records_to_preds(recs, conf_threshold=args.conf_threshold, masks="rle")
        videos.append((preds, opt_utils.track_planes(preds, cfg)))
        order.append((vid, recs))
    t0 = time.perf_counter()
    stats = opt_utils.Stats()
    outs = opt_utils.optimize_videos(videos, [args.seed + i for i in range(len(videos))], cfg=cfg,
                                     device=args.device, stats=stats)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    for (vid, recs), (preds, planes), out in zip(order, videos, outs):
        io.save_results(args.output, vid, io.opt_preds_to_records(out, recs), planes, masks=args.save_masks)
        if args.save_obj:
            for k in (0, len(preds) // 3, 2 * len(preds) // 3, len(preds) - 1):
                io.write_obj(os.path.join(args.output, f"{vid}_frame{k}.obj"), out, planes, k, cfg)
    if args.gt_json:
        import json
        from articulation3d_b200 import evaluation
        with open(args.gt_json) as f:
            gt = evaluation.CocoGT(json.load(f))
        before = [r for _, recs in order for r in io.opt_preds_to_records(
            io.records_to_preds(recs, conf_threshold=args.conf_threshold, masks="rle"), recs)]
        after = [r for (_, recs), out in zip(order, outs) for r in io.opt_preds_to_records(out, recs)]
        for tag, records in (("before", before), ("after", after)):
            res = evaluation.evaluate_for_arti_axis(records, gt, evaluation.Metadata(), 0.0)
            print(f"AP {tag} optimisation: " + ", ".join(f"{k} {float(v):.4f}" for k, v in res.items()))
    n_tracks = sum(len(p["rot"]) + len(p["trans"]) for _, p in videos)
    print(f"{len(videos)} video(s), {n_tracks} track(s): {stats.units_visited} track-frame x candidate evaluations "
          f"in {dt * 1e3:.1f} ms ({stats.passes} device passes) -> {args.output}")


if __name__ == "__main__":
    main()
