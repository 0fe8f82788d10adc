#!/usr/bin/env python
"""bench.py — RGBD frames/s integrated (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config C2|C3|C4|C5]
                    [--dump-outputs DIR]

Default workload = BASELINE.json configs[1] (C2: TUM1-shape 640x480, 5 mm voxels, tau 0.04 m, 300 synthetic frames
per step).  `--config C3` (Replica shape 1200x680 + class labels), `C4` (ScanNet shape, 4 mm, meant for 4 GPUs) and
`C5` (KITTI shape, 10 cm, meant for 8 GPUs, + mesh extraction) run the other configs.
One "step" = one pass of the hot path (hash allocation + projective TSDF/colour update) over the whole synthetic
sequence.  Warm-up passes populate the map; timed passes are steady state.  The volume runs the reference's Open3D
configuration (16^3 volume units, stride 4): results are bit-identical to the Open3D-order oracle.

  value     frames/s with the frames already resident in HBM, CUDA events on the launching stream, max over ranks.
  e2e       the same metric through the public API with PINNED HOST frames: `FrameIngest.integrate_batch` (every
            frame crosses PCIe once: rank r uploads 1/N of each chunk, NCCL all-gather over NVLink completes it,
            overlapped with the kernels) -> `b2v_integrate_batch`; one D2H read of the step's result per step.
  roofline  the dominant kernel of the timed region (`integrate_group_kernel`): achieved = bytes it MOVES
            (2*S*512 per block visit + 16 B per texel of the group's frames) / CUDA-event launch durations, against
            MEASURED_PEAKS.json; `per_frame_equivalent` is SURVEY.md 8d's formula (2*S*512*A_f + 7*W*H per frame,
            what frame-by-frame integration must move) over the same time.  `per_frame_kernel` gives the un-fused
            HBM-bound `integrate_kernel` warm (consecutive frames share L2-resident blocks) and cold (L2 flushed).
  cpu_baseline / --impl reference   the Open3D-order CPU port (oracle/open3d_order.c, OpenMP over volume units, the
            team size that a short probe finds fastest among 8 .. all host threads) on the same frames; Open3D
            itself is not installable here.

N > 1 (torchrun): the voxel-block hash space is sharded by BlockKeyHash % N; every rank integrates every frame into
the blocks it owns.  Total work is fixed ("strong" scaling).  The union of the shards is checked against an
unsharded volume on rank 0 by per-block checksums (`parity`).
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from pyslam_b200 import synthetic as S  # noqa: E402

METRIC = "rgbd_frames_per_sec_integrated"
UNIT = "frames/s"
VOXEL_RECORD_BYTES = 20  # tsdf f32 + weight f32 + rgb 3 x f32 (SURVEY.md §8d "S")
SHAPE_NAMES = {"C1": "plumbing", "C2": "TUM1-shape", "C3": "Replica-shape", "C4": "ScanNet-shape",
               "C5": "KITTI-00-shape", "T0": "test"}


# ------------------------------------------------------------------------------------------------
# synthetic workload
# ------------------------------------------------------------------------------------------------

def _render_one(args):
    name, i = args
    d, c, T = S.render_frame(S.CONFIGS[name], i)
    return i, d, c, T


def load_frames(cfg_name: str, n_frames: int, rank: int, world: int, barrier=None):
    """Render (rank 0, all cores) or load the cached frames of the sequence."""
    cfg = S.CONFIGS[cfg_name]
    n_frames = min(n_frames, cfg.n_frames)
    step = max(cfg.n_frames // n_frames, 1)
    idx = [k * step for k in range(n_frames)]
    cache = f"/tmp/b2v_frames_{cfg_name}_{n_frames}_{step}.npz"
    if rank == 0 and not os.path.exists(cache):
        import multiprocessing as mp
        procs = max(1, min(len(os.sched_getaffinity(0)), 48))
        with mp.get_context("fork").Pool(procs) as pool:
            res = sorted(pool.map(_render_one, [(cfg_name, i) for i in idx], chunksize=2))
        tmp = cache + f".tmp{os.getpid()}.npz"
        np.savez(tmp, depth=np.stack([r[1] for r in res]), color=np.stack([r[2] for r in res]),
                 Tcw=np.stack([r[3] for r in res]))
        os.replace(tmp, cache)
    if barrier is not None:
        barrier()
    z = np.load(cache)
    return cfg, z["depth"], z["color"], z["Tcw"]


# ------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md "clocks line")
# ------------------------------------------------------------------------------------------------

class ClockSampler:
    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(np.max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU arms (oracle = test infrastructure; this is one of the two places bench.py may run it)
# ------------------------------------------------------------------------------------------------

def host_threads() -> int:
    """Host threads this process may use (torchrun sets OMP_NUM_THREADS=1: the OpenMP team size is passed explicitly)."""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


CPU_PORT = ("Open3D-order CPU port (oracle/open3d_order.c: ScalableTSDFVolume(voxel, trunc, RGB8, 16, 4).integrate in "
            "Open3D's operation order; OpenMP over the touched 16^3 units where Open3D parallelises over x inside "
            "one unit at a time; gcc -O3 -ffp-contract=off like Open3D's FMA-less x86-64 wheels)")


def cpu_port_fps(cfg, depth, color, Tcw, n_sample, threads, passes=1):
    """Steady-state frames/s of the Open3D-order CPU port on a bounded sample."""
    import oracle
    orc = oracle.Open3DOrderVolume(cfg.voxel_size, cfg.sdf_trunc, 16, 4)
    n = min(n_sample, len(depth))
    for i in range(n):  # populate (allocation pass), untimed
        orc.integrate(depth[i], color[i], cfg.K, Tcw[i], cfg.depth_trunc, nthreads=threads)
    t0 = time.perf_counter()
    for _ in range(passes):
        for i in range(n):
            orc.integrate(depth[i], color[i], cfg.K, Tcw[i], cfg.depth_trunc, nthreads=threads)
    dt = time.perf_counter() - t0
    return passes * n / dt, n, passes


def best_thread_count(cfg, depth, color, Tcw) -> int:
    """The port's per-frame allocation pass is serial (as Open3D's is) and the box may be shared: pick the OpenMP
    team size with the best steady-state throughput on 8 frames, best of 3 rounds per candidate so that a burst of
    foreign load on the host does not pick a poor size (explicit num_threads: OMP_NUM_THREADS is ignored)."""
    import oracle
    hi = host_threads()
    cands = sorted({c for c in (8, 16, 32, 48, 64, 96, hi) if c <= hi} | {hi})
    orc = oracle.Open3DOrderVolume(cfg.voxel_size, cfg.sdf_trunc, 16, 4)
    n = min(8, len(depth))
    for i in range(n):
        orc.integrate(depth[i], color[i], cfg.K, Tcw[i], cfg.depth_trunc, nthreads=hi)
    best, best_t = hi, float("inf")
    for _ in range(3):
        for c in cands:
            t0 = time.perf_counter()
            for i in range(n):
                orc.integrate(depth[i], color[i], cfg.K, Tcw[i], cfg.depth_trunc, nthreads=c)
            dt = time.perf_counter() - t0
            if dt < best_t:
                best, best_t = c, dt
    return best


def frontend_points(cfg, d, c, T):
    """World points / colours the reference front-end hands to VoxelBlockGrid.integrate
    (pyslam/utilities/depth.py:45-85 + pyslam/dense/volumetric_integrator_voxel_grid.py:262-281)."""
    valid = (d > 0.0) & (d < cfg.depth_trunc)
    z = d[valid].astype(np.float64)
    rows, cols = np.where(valid)
    x = (cols - cfg.cx) * z / cfg.fx
    y = (rows - cfg.cy) * z / cfg.fy
    Twc = S.inv_T(T)
    R, t = Twc[:3, :3], Twc[:3, 3]
    pw = np.stack([x * R[a, 0] + y * R[a, 1] + z * R[a, 2] + t[a] for a in range(3)], axis=1)
    return pw.astype(np.float32), (c[valid] / 255.0).astype(np.float32)


def cpu_ref_grid_fps(cfg, depth, color, Tcw, n_sample):
    """frames/s of the UNMODIFIED reference VoxelBlockGrid::integrate (point-average grid; 1 core, sequential branch:
    oneTBB is absent) fed the world points the reference front-end derives from the same frames."""
    import oracle
    if not oracle.have_ref():
        return None
    g = oracle.RefGrid(cfg.voxel_size, 8)
    n = min(n_sample, len(depth))
    total, pts = 0.0, 0
    for i in range(n):
        p, col = frontend_points(cfg, depth[i], color[i], Tcw[i])
        total += g.integrate(p, col)
        pts += len(p)
    return n / total, pts / n, g.dump_blocks()


def grid_parity(cfg, depth, color, Tcw, n, ref_dump, device):
    """Full-size check of the point-average grid: the same n frames through b2v_grid_integrate_rgbd vs the unmodified
    compiled reference fed the reference front-end's points.  Keys and hashes must be equal; per-voxel counts may
    differ where a point lies within float rounding of a voxel face (the reference front-end's numpy arithmetic vs the
    fused kernel's: tests/test_gpu_grid.py), so the differing count is reported."""
    from pyslam_b200 import VoxelBlockGrid
    g = VoxelBlockGrid(cfg.voxel_size, 8, capacity_blocks=1 << 17, device=device)
    for i in range(n):
        g.integrate_rgbd(depth[i], color[i], cfg.K, S.inv_T(Tcw[i]), max_depth=cfg.depth_trunc)
    d = g.dump_blocks()
    g.close()

    def order(k):
        return np.lexsort((k[:, 2], k[:, 1], k[:, 0]))
    og, orf = order(d["keys"]), order(ref_dump["keys"])
    same_keys = len(og) == len(orf) and bool(np.array_equal(d["keys"][og], ref_dump["keys"][orf]))
    out = {"frames": n, "blocks_gpu": int(len(og)), "blocks_reference": int(len(orf)), "block_keys_equal": same_keys}
    if same_keys:
        out["hashes_equal"] = bool(np.array_equal(d["hashes"][og], ref_dump["hashes"][orf]))
        cg, cr = d["count"][og], ref_dump["count"][orf]
        out["voxels_gpu"] = int((cg > 0).sum())
        out["voxels_reference"] = int((cr > 0).sum())
        out["points_gpu"] = int(cg.sum())
        out["points_reference"] = int(cr.sum())
        out["voxels_with_a_different_count"] = int((cg != cr).sum())
    return out


# ------------------------------------------------------------------------------------------------
# arms
# ------------------------------------------------------------------------------------------------

def workload_config(cfg, frames_per_step, world, extra=None):
    out = {
        "workload": (f"{cfg.name} {SHAPE_NAMES.get(cfg.name, '')} {cfg.width}x{cfg.height} RGBD, voxel {cfg.voxel_size} m, "
                     f"sdf_trunc {cfg.sdf_trunc} m, depth_trunc {cfg.depth_trunc} m, block 8^3 in 16^3 Open3D volume "
                     f"units, alloc stride 4"),
        "frames_per_step": int(frames_per_step),
        "voxel_record_bytes": VOXEL_RECORD_BYTES,
        "parallelism": f"hash-shard x{world} (BlockKeyHash % N) + frame-split ingest (NCCL all-gather)" if world > 1
        else "single GPU",
    }
    if extra:
        out.update(extra)
    return out


def run_reference_arm(args, rank):
    if rank != 0:
        return
    cfg, depth, color, Tcw = load_frames(args.config, args.frames, 0, 1)
    import oracle
    threads = best_thread_count(cfg, depth, color, Tcw)
    orc = oracle.Open3DOrderVolume(cfg.voxel_size, cfg.sdf_trunc, 16, 4)
    # bounded sample: the whole sequence unless a step would take longer than ~12 s on this host
    t0 = time.perf_counter()
    for i in range(min(8, len(depth))):
        orc.integrate(depth[i], color[i], cfg.K, Tcw[i], cfg.depth_trunc, nthreads=threads)
    per_frame = (time.perf_counter() - t0) / min(8, len(depth))
    n_sample = int(max(8, min(len(depth), 12.0 / max(per_frame, 1e-6))))

    def one_step():
        for i in range(n_sample):
            orc.integrate(depth[i], color[i], cfg.K, Tcw[i], cfg.depth_trunc, nthreads=threads)

    for _ in range(max(min(args.warmup, 2), 1)):
        one_step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one_step()
    dt = time.perf_counter() - t0
    fps = args.steps * n_sample / dt
    sample = (f"first {n_sample} of the {len(depth)} frames of the {args.config} sequence per step, steady state; "
              + CPU_PORT)
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": workload_config(cfg, n_sample, 1),
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": sample, "cpu_model": cpu_model(), "host_threads": host_threads()},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def shard_checksum(dump):
    """Order-independent 64-bit checksum of a block dump: sum over blocks of (bit patterns of the planes, mixed
    with the block key)."""
    if len(dump["keys"]) == 0:
        return 0, 0
    bits = np.ascontiguousarray(dump["vox"]).view(np.uint32).astype(np.uint64)
    per_block = bits.reshape(bits.shape[0], -1).sum(axis=1, dtype=np.uint64)
    k = dump["keys"].astype(np.int64).astype(np.uint64)
    mix = (k[:, 0] * np.uint64(0x9E3779B97F4A7C15)) ^ (k[:, 1] * np.uint64(0xC2B2AE3D27D4EB4F)) ^ \
          (k[:, 2] * np.uint64(0x165667B19E3779F9))
    with np.errstate(over="ignore"):
        total = int(((per_block + np.uint64(1)) * (mix | np.uint64(1))).sum(dtype=np.uint64))
    return total, len(dump["keys"])


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, vol, suffix="", budget=DUMP_BYTES):
    """What a caller reads back from the volume after the last timed step, as .npy files in out_dir: the block count,
    and block keys (float64 [m,3]) with their tsdf, weight (float32 [m,512]) and rgb (float32 [m,3,512]) planes,
    sorted by key.  When all blocks would exceed `budget` bytes, m is a fixed seeded sample of them."""
    d = vol.dump_blocks()
    keys, vox = d["keys"], d["vox"]
    order = np.lexsort((keys[:, 2], keys[:, 1], keys[:, 0]))
    m = min(len(order), budget // (3 * 8 + vox.itemsize * int(np.prod(vox.shape[1:]))))
    if m < len(order):
        order = order[np.sort(np.random.default_rng(0).choice(len(order), m, replace=False))]
    keys, vox = keys[order], vox[order]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("num_blocks", np.array([len(d["keys"])], np.float64)), ("block_keys", keys.astype(np.float64)),
                    ("tsdf", vox[:, 0]), ("weight", vox[:, 1]), ("rgb", vox[:, 2:5])):
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), np.ascontiguousarray(a))


def run_gpu_arm(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # (NCCL_DEBUG is left to the caller: even WARN prints a version banner on stdout, and stdout is the JSON line)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()

    def all_max(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    from pyslam_b200 import B200TsdfVolume
    from pyslam_b200.sharding import FrameIngest
    cfg, depth, color, Tcw = load_frames(args.config, args.frames, rank, world, barrier)
    F, H, W = depth.shape
    shards = args.shard_of if (world == 1 and args.shard_of > 1) else world
    group = args.group if args.group > 0 else 32

    def make_volume(shard_rank, shard_count):
        v = B200TsdfVolume(cfg.voxel_size, cfg.sdf_trunc, cfg.depth_trunc, capacity_blocks=args.capacity,
                           device=local_rank, shard_rank=shard_rank, shard_count=shard_count)
        v.set_group_size(group)
        return v

    vol = make_volume(rank if world > 1 else 0, shards)
    # a dedicated (non-default) stream: the legacy default stream has handle 0, which the C ABI reads
    # as "use the library's own stream" and which torch events would not observe
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    d_dev = torch.from_numpy(depth).cuda()
    c_dev = torch.from_numpy(color).cuda()
    d_pin = torch.from_numpy(depth).pin_memory()
    c_pin = torch.from_numpy(color).pin_memory()
    K = cfg.K
    ingest = FrameIngest(vol, chunk_frames=args.chunk)

    def step_resident():
        # one C call enqueues the whole sequence (frames already in HBM) on torch's current stream
        vol.integrate_batch(d_dev, c_dev, K, Tcw, stream=stream.cuda_stream)

    def step_e2e():
        ingest.integrate_batch(d_pin, c_pin, K, Tcw)
        ingest.synchronize()
        return vol.last_frame_stats()  # D2H read of the step's result (the volume's counter block)

    # ---- the clock sampler starts first so that it is up (nvidia-smi takes ~0.2 s to deliver its first sample)
    #      when the timed regions run; the GPU stays under load until it delivers ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    t_load = time.perf_counter()
    while len(sampler.rows) < 2 and time.perf_counter() - t_load < 1.5:
        step_resident()
        torch.cuda.synchronize()
    # the loop above runs a varying number of steps: start the map again so that every run integrates the same
    # number of passes before the timed region ends (the outputs of --dump-outputs are then reproducible)
    vol.reset()

    # ---- warm-up (populates the map: steady state afterwards) ----
    for _ in range(max(args.warmup, 3)):
        step_resident()
    torch.cuda.synchronize()
    vol.synchronize()
    nb = vol.num_blocks()

    # ---- value: inputs resident in HBM, CUDA events on the launching stream ----
    barrier()
    torch.cuda.synchronize()
    for _ in range(2):
        step_resident()
    torch.cuda.synchronize()
    upd0, launches0 = vol.counters()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step_resident()
    e1.record(stream)
    torch.cuda.synchronize()
    barrier()
    ms_max = all_max(e0.elapsed_time(e1))
    upd1, launches1 = vol.counters()
    value = args.steps * F / (ms_max * 1e-3)
    if args.dump_outputs:
        # every rank writes its own shard: the 64 MB are shared out among the ranks
        dump_outputs(args.dump_outputs, vol, f"_rank{rank}" if world > 1 else "", DUMP_BYTES // world)

    # ---- e2e: pinned host frames through the public API, H2D (+ NVLink all-gather) inside the timed region ----
    for _ in range(2):
        step_e2e()
    barrier()
    torch.cuda.synchronize()
    h2d0, gat0 = ingest.h2d_bytes, ingest.gather_bytes
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    dt = all_max(time.perf_counter() - t0)
    e2e_value = args.steps * F / dt
    h2d_rank = (ingest.h2d_bytes - h2d0) / args.steps
    gather_rank = (ingest.gather_bytes - gat0) / args.steps
    t_load = time.perf_counter()
    while len(sampler.rows) < 6 and time.perf_counter() - t_load < 1.0:   # short runs: a few more samples under load
        step_resident()
        torch.cuda.synchronize()
    clocks = sampler.stop()  # sampled under load across the warm-up, the timed regions and the tail above

    # ---- roofline: CUDA events around every integrate launch over passes of the same work ----
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # 256 MiB > 126 MB L2

    def profile_pass(overlap, fusion, cold=False):
        vol.set_overlap(overlap)
        vol.set_fusion(fusion)
        vol.profile_enable(True)
        u0, _ = vol.counters()
        b0 = vol.block_visits()
        if cold:   # one frame per call, L2 flushed (256 MiB written) before each frame's kernels
            for i in range(0, F, max(F // 60, 1)):
                flush.zero_()
                vol.integrate(d_dev[i], c_dev[i], K, Tcw[i], stream=stream.cuda_stream)
        else:
            for _ in range(min(args.steps, 3)):
                step_resident()
        torch.cuda.synchronize()
        a_ms, i_ms, nfr, nl = vol.profile_read()
        u1, _ = vol.counters()
        b1 = vol.block_visits()
        vol.profile_enable(False)
        upd, vis = u1 - u0, b1 - b0
        survey_bytes = 2 * VOXEL_RECORD_BYTES * 512 * upd + 7 * W * H * nfr       # SURVEY.md §8d formula
        moved_bytes = 2 * VOXEL_RECORD_BYTES * 512 * vis + 16 * W * H * nfr        # blocks visited + texels
        sec = i_ms * 1e-3
        return dict(alloc_ms=a_ms, integ_ms=i_ms, frames=nfr, launches=nl, updates=upd, visits=vis,
                    survey_bytes=survey_bytes, moved_bytes=moved_bytes,
                    gbs=survey_bytes / sec / 1e9 if sec > 0 else 0.0,
                    moved_gbs=moved_bytes / sec / 1e9 if sec > 0 else 0.0)

    situ = profile_pass(True, True)      # the timed-region schedule: fused groups, allocate overlapped
    iso = profile_pass(False, False)     # one frame per launch, kernels serialised: warm L2 (consecutive frames)
    cold = profile_pass(False, False, cold=True)
    vol.set_overlap(True)
    vol.set_fusion(True)
    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    try:
        mp_ = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak, peak_src = float(mp_["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        pass
    traffic, traffic_note = None, None
    if world == 1 and args.config == "C2" and args.frames == 300 and shards == 1:
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "latest.json")))
            ent = prof.get("integrate_group_kernel", {})
            if ent.get("workload") == "C2x300":
                traffic = ent.get("dram_bytes_per_launch")
                traffic_note = ent.get("source")
        except Exception:
            pass

    # ---- parity evidence at N > 1: union of the shards == an unsharded volume (per-block checksums) ----
    parity = None
    if world > 1:
        n_par = min(F, 64)
        sv = make_volume(rank, world)
        sv.integrate_batch(d_dev[:n_par], c_dev[:n_par], K, Tcw[:n_par])
        cs, nblk = shard_checksum(sv.dump_blocks())
        sv.close()
        t = torch.tensor([cs & 0x7FFFFFFFFFFFFFFF, nblk], dtype=torch.int64, device="cuda")
        ts = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(ts, t)
        if rank == 0:
            uv = make_volume(0, 1)
            uv.integrate_batch(d_dev[:n_par], c_dev[:n_par], K, Tcw[:n_par])
            dump = uv.dump_blocks()
            uv.close()
            from pyslam_b200.sharding import owner_of
            own = owner_of(dump["keys"], world)
            ok = True
            for r in range(world):
                sel = own == r
                cr, nr = shard_checksum({"keys": dump["keys"][sel], "vox": dump["vox"][sel]})
                ok = ok and (cr & 0x7FFFFFFFFFFFFFFF) == int(ts[r][0].item()) and nr == int(ts[r][1].item())
            parity = {"frames": n_par, "blocks": int(len(dump["keys"])), "shards_equal_unsharded_volume": bool(ok),
                      "how": "per-rank checksum of (block key, bit patterns of the 5 planes) vs the same checksum of "
                             "rank 0's unsharded volume restricted to BlockKeyHash % N == r"}

    # ---- mesh extraction, reported separately (SURVEY.md 8d): marching cubes over the whole map ----
    mesh_info = None
    if world == 1:
        import ctypes as C
        nv_, nt_ = C.c_int64(0), C.c_int64(0)
        vol.synchronize()
        vol._L.b2v_extract_mesh(vol._h, C.byref(nv_), C.byref(nt_))   # warm-up (allocates scratch)
        t0 = time.perf_counter()
        vol._L.b2v_extract_mesh(vol._h, C.byref(nv_), C.byref(nt_))   # kernels + size read-back, no bulk copy
        mesh_ms = 1e3 * (time.perf_counter() - t0)
        mesh_bytes = 1.42 * VOXEL_RECORD_BYTES * 512 * nb + 24 * nv_.value + 12 * nt_.value
        mesh_info = {"ms_per_extract": mesh_ms, "vertices": int(nv_.value), "triangles": int(nt_.value),
                     "blocks": int(nb), "triangles_per_s": nt_.value / (mesh_ms * 1e-3),
                     "algorithmic_bytes": mesh_bytes, "gbs": mesh_bytes / (mesh_ms * 1e-3) / 1e9,
                     "frac_of_peak": mesh_bytes / (mesh_ms * 1e-3) / 1e9 / peak,
                     "note": "b2v_extract_mesh on the populated map: neighbours, classify, scan, vertices, "
                             "triangles kernels + a 8-byte size read-back; arrays stay on the device; wall clock"}
    elif args.config == "C5" or args.mesh:
        from pyslam_b200 import sharding
        sharding.extract_mesh_distributed(vol, dst=0)   # warm-up: NCCL point-to-point set-up, scratch allocations
        barrier()
        t0 = time.perf_counter()
        m = sharding.extract_mesh_distributed(vol, dst=0)
        barrier()
        mesh_ms = 1e3 * (time.perf_counter() - t0)
        if rank == 0:
            mesh_info = {"ms_per_extract": mesh_ms, "vertices": int(len(m.vertices)), "triangles": int(len(m.triangles)),
                         "note": f"{world}-GPU spatial shards gathered GPU-to-GPU over NCCL onto rank 0, marching cubes "
                                 f"there, arrays copied to the host (wall clock, includes the gather)"}

    # ---- secondary e2e figure: the same frames as RAW 16-bit depth (TUM-style payload, 5000 units per metre) ----
    e2e_u16 = None
    if args.config in ("C2", "C4"):
        scale = np.float32(1.0 / 5000.0)
        raw16 = torch.from_numpy(np.round(depth * 5000.0).astype(np.uint16)).pin_memory()
        for _ in range(2):
            ingest.integrate_batch(raw16, c_pin, K, Tcw, depth_scale=scale)
            ingest.synchronize()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            ingest.integrate_batch(raw16, c_pin, K, Tcw, depth_scale=scale)
            ingest.synchronize()
        dt16 = all_max(time.perf_counter() - t0)
        e2e_u16 = {"value": args.steps * F / dt16, "unit": UNIT, "h2d_bytes_per_step": int(F * H * W * 5),
                   "d2h_bytes_per_step": 256,
                   "api": "FrameIngest.integrate_batch(depths uint16, colors, K, poses, depth_scale) -> "
                          "b2v_integrate_batch_u16: raw 16-bit depth over PCIe (and NVLink), widened to float32 metres "
                          "on the GPU (bit-identical to depth.astype(float32) * depth_factor on the host)"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- extra legs (rank 0, N = 1 only) ----
    cpu = None
    extra = {}
    if world == 1 and not args.no_cpu:
        threads = best_thread_count(cfg, depth, color, Tcw)
        fps, n_s, passes = cpu_port_fps(cfg, depth, color, Tcw, args.cpu_frames, threads)
        cpu = {"value": fps, "unit": UNIT, "cores": threads, "kind": "port", "cpu_model": cpu_model(),
               "host_threads": host_threads(),
               "sample": f"first {n_s} frames of the sequence, {passes} steady-state pass(es); " + CPU_PORT}
        fps1, _, _ = cpu_port_fps(cfg, depth, color, Tcw, min(args.cpu_frames, 8), 1, passes=1)
        extra["cpu_baseline_1core"] = {"value": fps1, "unit": UNIT, "cores": 1, "kind": "port"}
        extra["point_average_grid"] = grid_leg(cfg, depth, color, Tcw, d_dev, c_dev, peak, local_rank)
        if cfg.n_classes > 0:
            extra["semantic_grid"] = semantic_leg(cfg, depth, color, Tcw, local_rank)

    n_l = max(situ["launches"], 1)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_max / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(cfg, F, world, {
            "blocks_in_map": int(nb), "active_blocks_per_frame": situ["updates"] / max(situ["frames"], 1),
            "frames_per_fused_group": group,
            "l2": (f"no flush in the timed region: each step streams {nb * 10240 / 1e6:.0f} MB of voxel blocks "
                   f"(> 126 MB L2) between two visits of the same block"),
            "timing": "CUDA events on the launching stream, max over ranks"}),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(F * H * W * 7),
                "h2d_bytes_per_step_per_rank": int(h2d_rank), "nvlink_gather_bytes_per_step_per_rank": int(gather_rank),
                "d2h_bytes_per_step": 256, "timing": "wall clock around a full device sync, max over ranks",
                "api": "FrameIngest.integrate_batch(depths, colors, K, poses) [pinned host frames; rank r uploads 1/N of "
                       "every chunk, NCCL all-gather over NVLink] -> B200TsdfVolume.integrate_batch -> b2v_integrate_batch"},
        **({"e2e_u16_depth": e2e_u16} if e2e_u16 else {}),
        "gpu_launches": int(launches1 - launches0),
        "roofline": {
            "kernel": f"integrate_group_kernel (up to {group} frames applied per block visit)", "bound": "hbm",
            "achieved": situ["moved_gbs"], "peak": peak, "peak_source": peak_src, "unit": "GB/s",
            "frac": situ["moved_gbs"] / peak if peak else None,
            "traffic": traffic, "traffic_source": traffic_note,
            "bytes_moved_per_launch": situ["moved_bytes"] / n_l,
            "avg_launch_us": 1e3 * situ["integ_ms"] / n_l,
            "frames_per_launch": situ["frames"] / n_l,
            "block_visits_per_update": situ["visits"] / max(situ["updates"], 1),
            "per_frame_equivalent": {
                "gbs": situ["gbs"], "frac": situ["gbs"] / peak if peak else None,
                "algorithmic_bytes_per_launch": situ["survey_bytes"] / n_l,
                "note": "SURVEY.md 8d formula 2*S*512*A_f + 7*W*H summed over the frames of a launch = what "
                        "frame-by-frame integration must move; the fused kernel reads / writes a block once per group, "
                        "so this is NOT bytes it moves (it is limited by instruction issue, see profiles/)"},
            "measured": "in situ: CUDA events around every launch in the timed-region schedule "
                        "(allocate kernels of the next group run beside it)",
            "allocate_group_kernel_avg_us_in_situ": 1e3 * situ["alloc_ms"] / n_l,
            "per_frame_kernel": {
                "kernel": "integrate_kernel (one frame per launch, b2v_set_fusion 0, b2v_set_overlap 0)",
                "bound": "hbm",
                "warm_l2": {"achieved": iso["gbs"], "frac": iso["gbs"] / peak if peak else None,
                            "avg_launch_us": 1e3 * iso["integ_ms"] / max(iso["launches"], 1),
                            "note": "consecutive frames: most of a frame's blocks are still in the 126 MB L2"},
                "cold_l2": {"achieved": cold["gbs"], "frac": cold["gbs"] / peak if peak else None,
                            "avg_launch_us": 1e3 * cold["integ_ms"] / max(cold["launches"], 1),
                            "note": "256 MiB written between frames: every block comes from HBM"},
                "allocate_kernel_avg_us": 1e3 * iso["alloc_ms"] / max(iso["frames"], 1)}},
        "clocks": clocks,
        **({"parity": parity} if parity else {}),
        **({"diagnostic": f"--shard-of {args.shard_of}: this process is rank 0 of a {args.shard_of}-way sharded job "
                          f"(value = that job's per-rank rate = its whole-job rate, ranks share nothing)"}
           if (world == 1 and args.shard_of > 1) else {}),
        "mesh": mesh_info,
        "cpu_baseline": cpu,
        **extra,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def grid_leg(cfg, depth, color, Tcw, d_dev, c_dev, peak, device):
    """The point-average voxel grid (cpp/volumetric's own model): b2v_grid_integrate_rgbd on the same frames vs the
    UNMODIFIED compiled reference VoxelBlockGrid::integrate_raw (the one comparison against real reference code)."""
    from pyslam_b200 import VoxelBlockGrid
    n = min(len(depth), 64)
    g = VoxelBlockGrid(cfg.voxel_size, 8, capacity_blocks=1 << 17, device=device)
    K4 = np.array(cfg.K, np.float64)
    Twc = [np.ascontiguousarray(S.inv_T(Tcw[i])).reshape(16) for i in range(n)]
    mx = float(cfg.depth_trunc)

    def one_pass():
        for i in range(n):
            rc = g._L.b2v_grid_integrate_rgbd(g._h, d_dev[i].data_ptr(), c_dev[i].data_ptr(), depth.shape[1],
                                              depth.shape[2], K4.ctypes.data, Twc[i].ctypes.data, mx, 0.0, 0)
            assert rc == 0
        g._check(g._L.b2v_grid_synchronize(g._h), "sync")

    one_pass()
    t0 = time.perf_counter()
    one_pass()
    dt = time.perf_counter() - t0
    pts = float(np.mean([((depth[i] > 0) & (depth[i] < cfg.depth_trunc)).sum() for i in range(n)]))
    out = {"gpu": {"value": n / dt, "unit": UNIT, "frames": n, "points_per_frame": pts,
                   "api": "b2v_grid_integrate_rgbd (device frames): depth2pointcloud + world transform + integrate",
                   "algorithmic_bytes_per_frame": 80 * pts, "gbs": 80 * pts * n / dt / 1e9,
                   "frac_of_peak": 80 * pts * n / dt / 1e9 / peak,
                   "bound": "L2 atomics (7 float / int atomics per point); 80 B / point is SURVEY.md 8d's figure"}}
    g.close()
    ref = cpu_ref_grid_fps(cfg, depth, color, Tcw, 6)
    if ref is not None:
        out["cpu_reference"] = {"value": ref[0], "unit": UNIT, "cores": 1, "kind": "reference", "frames": 6,
                                "sample": "6 frames, unmodified cpp/volumetric VoxelBlockGrid::integrate_raw<float,float> "
                                          "(sequential branch: oneTBB is not installed; g++ -O3 -march=x86-64-v3), fed "
                                          "the front-end's world points (not timed)"}
        out["speedup_vs_reference_1core"] = out["gpu"]["value"] / ref[0]
        out["parity"] = grid_parity(cfg, depth, color, Tcw, 6, ref[2], device)
    return out


def semantic_leg(cfg, depth, color, Tcw, device):
    """C3: label fusion per voxel (VoxelBlockSemanticProbabilisticGrid) through the fused RGBD front-end."""
    from pyslam_b200 import VoxelBlockSemanticProbabilisticGrid
    n = min(len(depth), 16)
    labels = [S.render_class_ids(cfg, i * max(cfg.n_frames // len(depth), 1)) for i in range(n)]
    g = VoxelBlockSemanticProbabilisticGrid(0.015, 8, capacity_blocks=1 << 16, device=device)
    t_all = []
    for rep in range(2):
        t0 = time.perf_counter()
        for i in range(n):
            g.integrate_rgbd(depth[i], color[i], cfg.K, S.inv_T(Tcw[i]), class_image=labels[i],
                             max_depth=cfg.depth_trunc)
        t_all.append(time.perf_counter() - t0)
    g.close()
    return {"value": n / t_all[1], "unit": UNIT, "ms_per_frame": 1e3 * t_all[1] / n, "frames": n,
            "api": "VoxelBlockSemanticProbabilisticGrid.integrate_rgbd (host frames + int32 class image in, synchronous): "
                   "depth2pointcloud + Bayesian label fusion at 1.5 cm voxels (the reference's default)",
            "note": "per-call host staging included"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C2", choices=["C2", "C3", "C4", "C5", "C1", "T0"])
    ap.add_argument("--frames", type=int, default=300, help="frames per step (the sequence length)")
    ap.add_argument("--capacity", type=int, default=1 << 19, help="block-pool capacity (10 KiB each)")
    ap.add_argument("--cpu-frames", type=int, default=32, help="frames in the bounded CPU sample")
    ap.add_argument("--group", type=int, default=0, help="frames per fused group (0: 32; the library default is 16)")
    ap.add_argument("--chunk", type=int, default=64, help="frames per ingest chunk (upload + all-gather granularity)")
    ap.add_argument("--mesh", action="store_true", help="N > 1: also time the distributed mesh extraction")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--shard-of", type=int, default=0,
                    help="diagnostic (N=1 only): act as rank 0 of a --shard-of-way sharded job on one GPU; ranks share "
                         "nothing, so this is the per-rank work of that job")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the volume they built to DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU volume; --impl reference has none")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    run_gpu_arm(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
