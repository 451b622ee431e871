"""Parity of ShardedRecording over NCCL: run under torchrun with N ranks (the product CudaEngine); every rank feeds its
share of a recording of full-size frames (2048 spokes x 1024 bins x 3 gains), rank 0 also runs RecordingDetection over
all frames on one GPU and compares points, labels, core flags and cluster counts id for id.

    torchrun --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29543 tools/check_sharded_recording.py [frames_per_rank] [eps_time] [min_frames]
"""
import os
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np
import torch
import torch.distributed as dist

from radar_point_cloud_tracking_b200 import device as dev, synthetic as syn
from radar_point_cloud_tracking_b200.pipeline import DetectionConfig
from radar_point_cloud_tracking_b200.recording import RecordingDetection
from radar_point_cloud_tracking_b200.sharded import ShardedRecording, split_frames

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
device = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=device)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 8
eps_time = float(sys.argv[2]) if len(sys.argv) > 2 else 2.0
min_frames = int(sys.argv[3]) if len(sys.argv) > 3 and int(sys.argv[3]) > 0 else None
n_frames = B * world + world // 2                                   # uneven shares
spec = syn.SweepSpec(seed=31, frames=n_frames, spokes=2048, bins=1024)
cfg = DetectionConfig(eps_time=eps_time, min_frames=min_frames)
ids = np.arange(n_frames) * 2 + 5
a, b = split_frames(n_frames, world, rank)
sr = ShardedRecording(cfg, rank, world, max_window_points=None)
c, s, r = (torch.from_numpy(t).to(device) for t in sr.pipe.spoke_tables(spec.angle_units(), spec.scale(), n_frames, spec.bins))
G = len(spec.gains)
for x in range(a, b, 4):                                            # blocks of 4 frames
    y = min(x + 4, b)
    sr.add_block(dev.synth_echo(spec, x, y - x, device=device), c[x * G:y * G], s[x * G:y * G], r[x * G:y * G], ids[x:y])
res = sr.finish()
n = res.points.n
mine = {"x": res.points.x[:n].cpu().numpy(), "labels": res.labels.cpu().numpy(), "core": res.core.cpu().numpy(),
        "ncl": res.n_clusters, "built": res.frames_built, "isum": res.isum.cpu().numpy() if res.isum is not None else None}
gathered = [None] * world
dist.gather_object(mine, gathered if rank == 0 else None, dst=0)
ok = True
if rank == 0:
    rec = RecordingDetection(cfg, local)
    for x in range(0, n_frames, 16):
        y = min(x + 16, n_frames)
        rec.add_block(dev.synth_echo(spec, x, y - x, device=device), c[x * G:y * G], s[x * G:y * G], r[x * G:y * G], ids[x:y])
    ref = rec.finish()
    m = ref.points.n
    ok = (np.array_equal(np.concatenate([g["x"] for g in gathered]), ref.points.x[:m].cpu().numpy())
          and np.array_equal(np.concatenate([g["labels"] for g in gathered]), ref.labels.cpu().numpy())
          and np.array_equal(np.concatenate([g["core"] for g in gathered]), ref.core.cpu().numpy())
          and all(g["ncl"] == ref.n_clusters and g["built"] == ref.frames_built for g in gathered)
          and all((g["isum"] is None) == (ref.isum is None) for g in gathered)
          and (ref.isum is None or all(g["isum"].tobytes() == ref.isum.cpu().numpy().tobytes() for g in gathered)))
    print(f"sharded recording x{world} (eps_time {eps_time}, min_frames {min_frames}): {n_frames} frames, {m} points, "
          f"{ref.n_clusters} clusters -> {'IDENTICAL to one GPU' if ok else 'MISMATCH'}")
flag = torch.tensor([1 if ok else 0], device=device)
dist.broadcast(flag, src=0)
dist.destroy_process_group()
sys.exit(0 if int(flag.item()) else 1)
