"""Temporal optimisation of saved predictions — the B200 counterpart of the reference's
``tools/opt_arti.py`` for the stage in scope (the detector is not re-run):

    python -m articulation3d_b200.tools.opt_arti --input instances_predictions.pth --output out/ [--save-obj] [--save-masks]
    torchrun --nnodes 1 --nproc-per-node 8 -m articulation3d_b200.tools.opt_arti --input ... --output out/

Reads the per-frame prediction records (RLE masks stay run-length encoded and are decoded on
the GPU), groups them by video, runs ``track_planes`` + ``optimize_planes('3dc')`` for all videos
in lock-step, and writes per video ``<id>_predictions_opt.pth`` (records as
tools/opt_arti.py:229-249), ``<id>_tracks.json`` (fitted axis + angle-per-frame track) and
optionally ``<id>_frame<k>.obj``; ``--save-masks`` adds every fitted frame's registered mask to the tracks JSON
as COCO RLE.  ``--synthetic N`` writes a synthetic input first (masks encoded on the tool's GPU; under torchrun
rank 0 writes it on its own).  The camera is the reference's 640x480 one scaled to the records' frame size
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
    ap.add_argument("--tracks", type=int, default=4)
    ap.add_argument("--frames", type=int, default=60)
    args = ap.parse_args(argv)

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


def _run(args, rank: int, world: int, device: torch.device):
    if args.synthetic and rank == 0:
        records = []
        for v in range(args.synthetic):
            preds, _ = synth.make_video(args.seed + v, args.tracks, args.frames)
            records += io.preds_to_records(preds, video_id=f"synthetic{v:02d}_0_0", start_image_id=v * 10000,
                                           device=device)
        torch.save(records, args.input)
    if world > 1:
        dist.barrier()

    # every rank reads the whole file (mapped, so the ranks share its pages) and sees the same video order
    order = list(adapter.group_by_video(adapter.load_predictions(args.input, mmap=world > 1)).items())
    cfg = frame_config(dict(order))
    mine = a3d_dist.shard_range(len(order), rank, world)
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
