"""Per-rank timing of an N-way hash-sharded job on ONE GPU (ranks share nothing, so rank 0 of N does that job's
per-rank work): frames/s and period per group of 8 frames.  Usage: python tools/shard_timeline.py [N]   (DESIGN.md §7)"""
import os, sys, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyslam_b200 import B200TsdfVolume
import bench
shards = int(sys.argv[1]) if len(sys.argv) > 1 else 8
cfg, depth, color, Tcw = bench.load_frames("C2", 64, 0, 1)
vol = B200TsdfVolume(cfg.voxel_size, cfg.sdf_trunc, cfg.depth_trunc, capacity_blocks=1<<19, shard_rank=0, shard_count=shards)
st = torch.cuda.Stream(); torch.cuda.set_stream(st)
d = torch.from_numpy(depth).cuda(); c = torch.from_numpy(color).cuda()
for _ in range(3): vol.integrate_batch(d, c, cfg.K, Tcw, stream=st.cuda_stream)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
t0 = time.perf_counter()
e0.record(st)
for _ in range(5): vol.integrate_batch(d, c, cfg.K, Tcw, stream=st.cuda_stream)
t_enq = time.perf_counter() - t0
e1.record(st); torch.cuda.synchronize()
ms = e0.elapsed_time(e1)
print(f"shards {shards}: {5*64/ms*1e3:.0f} frames/s, {ms/5/8*1e3:.1f} us per group of 8; host enqueue {t_enq/5/8*1e6:.1f} us per group")
vol.profile_enable(True)
vol.integrate_batch(d, c, cfg.K, Tcw, stream=st.cuda_stream)
torch.cuda.synchronize()
print(vol.profile_read())
