"""Temporal optimisation of saved predictions — the B200 counterpart of the reference's
``tools/opt_arti.py`` for the stage in scope (the detector is not re-run):

    python -m articulation3d_b200.tools.opt_arti --input instances_predictions.pth --output out/ [--save-obj] [--save-masks] \
        [--save-video [--fps 30] [--image-root DIR]] [--save-depth]
    torchrun --nnodes 1 --nproc-per-node 8 -m articulation3d_b200.tools.opt_arti --input ... --output out/

Reads the per-frame prediction records (RLE masks stay run-length encoded and are decoded on
the GPU), groups them by video, runs ``track_planes`` + ``optimize_planes('3dc')`` for all videos
in lock-step, and writes per video ``<id>_predictions_opt.pth`` (records as
tools/opt_arti.py:229-249), ``<id>_tracks.json`` (fitted axis + angle-per-frame track) and
optionally ``<id>_frame<k>.obj``; ``--save-masks`` adds every fitted frame's registered mask to the tracks JSON
as COCO RLE; ``--save-video`` writes ``<id>.mp4``, every frame drawn with the fitted result (``render.write_video``)
over ``--image-root``/<record file_name> (flat grey without it; missing or wrongly sized images stop the tool before
any device work); ``--save-depth`` writes ``<id>_depth/<k:05d>.png`` (per-frame depth of the fitted planes, uint16
millimetres, 0 = no plane) and ``<id>_normals.mp4`` (their surface normals; ``render.write_plane_maps``, detections
gated by ``--conf-threshold``).  ``--override-depth`` first replaces every instance's plane offset by the one its record's
``pred_depth`` implies (the reference's ``override_depth``), streamed through the GPU per rank.  ``--synthetic N``
writes a synthetic input first (masks encoded on the tool's GPU; under torchrun rank 0 writes it on its own;
``--synthetic-depth`` adds a rendered ``pred_depth``).  The camera is the reference's 640x480 one scaled to the records' frame size
(``segmentation.size``).

Under torchrun (WORLD_SIZE > 1) rank r runs on cuda:$LOCAL_RANK and converts, tracks, optimises and writes
the contiguous block of videos ``dist.shard_range`` gives it (the reference's SLURM split); video i keeps
seed ``--seed + i``, so every output file equals a one-GPU run's.  Rank 0 prints the AP table over all
videos and the summary line (sums over ranks, the slowest rank's optimise time).
"""
from __future__ import annotations

import argparse
import functools
import os
import time

import torch
import torch.distributed as dist

from articulation3d_b200 import OptConfig, adapter, io, opt_utils, synth
from articulation3d_b200 import dist as a3d_dist


def frame_index(record) -> int:
    """Trailing integer of the file name (``<yt id>_<shot>_<frame>_<offset>.png``)."""
    stem = os.path.splitext(os.path.basename(record["file_name"]))[0]
    return int(stem.split("_")[-1])


def frame_config(groups) -> OptConfig:
    """``OptConfig`` of the frame size (H, W) the records' masks carry (``segmentation.size``): ``OptConfig()`` at
    640x480 (and when no record has a mask), else ``OptConfig.scaled(W, H)``.  Raises ``ValueError`` when the
    masks of ``groups`` (video id -> records) differ in size."""
    first = None
    for vid, recs in groups.items():
        for r in recs:
            for inst in r["instances"]:
                seg = inst.get("segmentation")
                if seg is None:
                    continue
                size = tuple(int(x) for x in seg["size"])
                if first is None:
                    first = (size, vid)
                elif size != first[0]:
                    raise ValueError(f"the records mix frame sizes: {list(first[0])} in video {first[1]}, "
                                     f"{list(size)} in video {vid}; give videos of one size per input file")
    H, W = first[0] if first else (480, 640)
    return OptConfig() if (H, W) == (480, 640) else OptConfig.scaled(W, H)


def _read_rgb(path: str):
    import cv2
    img = cv2.imread(path, cv2.IMREAD_COLOR) if os.path.isfile(path) else None
    return None if img is None else cv2.cvtColor(img, cv2.COLOR_BGR2RGB)


def check_images(root: str, order, cfg: OptConfig):
    """Every record's ``root/<file_name>`` must be a readable image of the records' frame size; SystemExit with
    the first offender otherwise.  Every rank checks every video, so a bad image stops all ranks alike."""
    for _, recs in order:
        for r in recs:
            path = os.path.join(root, r["file_name"])
            img = _read_rgb(path)
            if img is None:
                raise SystemExit(f"--image-root: cannot read {path}")
            if img.shape[:2] != (cfg.height, cfg.width):
                raise SystemExit(f"--image-root: {path} is {img.shape[1]}x{img.shape[0]}, the records' frames are "
                                 f"{cfg.width}x{cfg.height}")


def load_images(root: str, recs):
    """(T, H, W, 3) uint8 RGB backgrounds of one video's records, in frame order."""
    import numpy as np
    return np.stack([_read_rgb(os.path.join(root, r["file_name"])) for r in recs])


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--input", required=True)
    ap.add_argument("--output", required=True)
    ap.add_argument("--conf-threshold", type=float, default=0.7)
    ap.add_argument("--seed", type=int, default=2020, help="per-video RNG seed base (tools/inference.py:172)")
    ap.add_argument("--device", default=None, help="default cuda:0; not accepted under torchrun")
    ap.add_argument("--save-obj", action="store_true")
    ap.add_argument("--save-masks", action="store_true", help="registered masks (COCO RLE) in the tracks JSON")
    ap.add_argument("--gt-json", default=None, help="COCO-style ground truth: print the AP table before / after "
                    "optimisation (tools/opt_arti.py:275-283)")
    ap.add_argument("--synthetic", type=int, default=0, help="first write N synthetic videos to --input "
                    "(masks encoded on the tool's GPU; under torchrun rank 0 writes)")
    ap.add_argument("--synthetic-depth", action="store_true", help="with --synthetic: the records carry a "
                    "rendered pred_depth (synth.render_depths)")
    ap.add_argument("--override-depth", action="store_true", help="replace every instance's plane offset by the "
                    "mean over its mask of normal . XYZ of the record's pred_depth before tracking "
                    "(adapter.override_depth_records; tools/inference.py:220, tools/opt_arti.py:173-185)")
    ap.add_argument("--save-video", action="store_true", help="<output>/<video id>.mp4 of the fitted result")
    ap.add_argument("--fps", type=float, default=30)
    ap.add_argument("--image-root", default=None, help="with --save-video: frame t is drawn over "
                    "DIR/<record file_name> instead of a flat grey image")
    ap.add_argument("--save-depth", action="store_true", help="<output>/<video id>_depth/<k>.png (uint16 mm) and "
                    "<video id>_normals.mp4 of the fitted planes")
    ap.add_argument("--tracks", type=int, default=4)
    ap.add_argument("--frames", type=int, default=60)
    args = ap.parse_args(argv)
    if args.synthetic_depth and not args.synthetic:
        ap.error("--synthetic-depth needs --synthetic N")
    if args.image_root and not args.save_video:
        ap.error("--image-root needs --save-video")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1:
        return _run(args, 0, 1, torch.device(args.device or "cuda:0"))
    if args.device is not None:
        ap.error(f"--device cannot be used under torchrun (WORLD_SIZE={world}): "
                 "every rank runs on cuda:$LOCAL_RANK")
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    try:
        _run(args, dist.get_rank(), world, dev)
    finally:
        dist.destroy_process_group()


def _override_depth(args, order, mine, rank: int, world: int, device: torch.device):
    """``adapter.override_depth_records`` of this rank's block of videos, in place.  Every rank checks every record
    first, so a bad record anywhere stops all ranks before any device work.  With ``--gt-json`` under torchrun,
    rank 0 receives the other blocks' new planes (one gather) for its "before" table.  Rank 0 prints frames,
    instances and depth bytes over all ranks, and the slowest rank's override time."""
    adapter.check_depth_records([r for _, recs in order for r in recs])
    block = [r for i in mine for r in order[i][1]]
    t0 = time.perf_counter()
    adapter.override_depth_records(block, device)           # ends in a D2H copy of the results
    dt = time.perf_counter() - t0
    counts = [len(block), sum(len(r["instances"]) for r in block),
              sum(r["pred_depth"].numel() * 4 for r in block if r["instances"])]
    where = ""
    if world > 1:
        total = torch.tensor(counts, dtype=torch.int64, device=device)
        dist.all_reduce(total)
        slowest = torch.tensor([dt], dtype=torch.float64, device=device)
        dist.all_reduce(slowest, op=dist.ReduceOp.MAX)
        counts, dt, where = total.tolist(), slowest.item(), f" on {world} GPUs"
        if args.gt_json:
            local = torch.cat([torch.zeros(0, 3)] + [r["pred_plane"].to(torch.float32) for r in block])
            local = local.view(torch.int32)
            if dist.get_backend() == "nccl":
                local = local.to(device)
            rows = a3d_dist.all_gather_rows(local).cpu().view(torch.float32)
            if rank == 0:
                k = 0
                for _, recs in order:
                    for r in recs:
                        n = len(r["instances"])
                        if n:
                            r["pred_plane"] = rows[k:k + n].clone()
                        k += n
    if rank == 0:
        frames, instances, nbytes = counts
        print(f"override-depth: {frames} frame(s), {instances} instance(s), {nbytes / 1e6:.1f} MB of depth "
              f"in {dt * 1e3:.1f} ms{where}")


def _run(args, rank: int, world: int, device: torch.device):
    if args.synthetic and rank == 0:
        records = []
        for v in range(args.synthetic):
            preds, scene = synth.make_video(args.seed + v, args.tracks, args.frames)
            depths = synth.render_depths(scene) if args.synthetic_depth else None
            records += io.preds_to_records(preds, video_id=f"synthetic{v:02d}_0_0", start_image_id=v * 10000,
                                           device=device, depths=depths)
        torch.save(records, args.input)
    if world > 1:
        dist.barrier()

    # every rank reads the whole file (mapped, so the ranks share its pages) and sees the same video order
    order = list(adapter.group_by_video(adapter.load_predictions(args.input, mmap=world > 1)).items())
    cfg = frame_config(dict(order))
    mine = a3d_dist.shard_range(len(order), rank, world)
    if args.image_root:
        check_images(args.image_root, order, cfg)
    if args.override_depth:
        _override_depth(args, order, mine, rank, world, device)
    videos = [None] * len(order)                  # only this rank's block is converted and tracked
    for i in mine:
        preds = io.records_to_preds(order[i][1], conf_threshold=args.conf_threshold, masks="rle")
        videos[i] = (preds, opt_utils.track_planes(preds, cfg))
    seeds = [args.seed + i for i in range(len(order))]
    t0 = time.perf_counter()
    stats = opt_utils.Stats()
    if world > 1:
        optimize_fn = functools.partial(opt_utils.optimize_videos, stats=stats)
        outs, _, _, _ = a3d_dist.optimize_videos_sharded(videos, seeds, cfg=cfg, device=device,
                                                         optimize_fn=optimize_fn)
    else:                                         # one process: no record tables to pack and gather
        outs = opt_utils.optimize_videos(videos, seeds, cfg=cfg, device=device, stats=stats)
    torch.cuda.synchronize(device)
    dt = time.perf_counter() - t0
    for i, out in zip(mine, outs):
        (vid, recs), (preds, planes) = order[i], videos[i]
        io.save_results(args.output, vid, io.opt_preds_to_records(out, recs), planes, masks=args.save_masks)
        if args.save_obj:
            for k in (0, len(preds) // 3, 2 * len(preds) // 3, len(preds) - 1):
                io.write_obj(os.path.join(args.output, f"{vid}_frame{k}.obj"), out, planes, k, cfg)
        if args.save_video:
            from articulation3d_b200 import render
            images = load_images(args.image_root, recs) if args.image_root else None
            render.write_video(os.path.join(args.output, f"{vid}.mp4"), out, planes, images=images, fps=args.fps,
                               cfg=cfg, device=device, score_thresh=args.conf_threshold)
        if args.save_depth:
            from articulation3d_b200 import render
            render.write_plane_maps(args.output, vid, out, planes, fps=args.fps, cfg=cfg, device=device,
                                    score_thresh=args.conf_threshold)
    if args.gt_json:
        if world == 1:
            after = [r for i, out in zip(mine, outs) for r in io.opt_preds_to_records(out, order[i][1])]
        else:
            dist.barrier()                        # every rank's files are written: they hold the "after" records
            after = [r for vid, _ in order for r in adapter.load_predictions(
                os.path.join(args.output, f"{vid}_predictions_opt.pth"), mmap=True)] if rank == 0 else None
        if rank == 0:
            import json
            from articulation3d_b200 import evaluation
            with open(args.gt_json) as f:
                gt = evaluation.CocoGT(json.load(f))
            before = [r for _, recs in order for r in io.opt_preds_to_records(
                io.records_to_preds(recs, conf_threshold=args.conf_threshold, masks="rle"), recs)]
            for tag, records in (("before", before), ("after", after)):
                res = evaluation.evaluate_for_arti_axis(records, gt, evaluation.Metadata(), 0.0)
                print(f"AP {tag} optimisation: " + ", ".join(f"{k} {float(v):.4f}" for k, v in res.items()))
    n_tracks = sum(len(videos[i][1]["rot"]) + len(videos[i][1]["trans"]) for i in mine)
    counts = [len(mine), n_tracks, stats.units_visited, stats.passes]
    where = ""
    if world > 1:
        total = torch.tensor(counts, dtype=torch.int64, device=device)
        dist.all_reduce(total)
        slowest = torch.tensor([dt], dtype=torch.float64, device=device)
        dist.all_reduce(slowest, op=dist.ReduceOp.MAX)
        counts, dt, where = total.tolist(), slowest.item(), f" on {world} GPUs"
    if rank == 0:
        n_videos, n_tracks, units, passes = counts
        print(f"{n_videos} video(s), {n_tracks} track(s): {units} track-frame x candidate evaluations "
              f"in {dt * 1e3:.1f} ms ({passes} device passes) -> {args.output}{where}")


if __name__ == "__main__":
    main()
