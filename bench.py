#!/usr/bin/env python
"""bench.py -- frames/sec at 1920x1080 (palette-index bit-exact vs the oracle) and the other BASELINE.json configs.

    python bench.py --gpus N --steps K --warmup W                 # configs[1]: this repo's CUDA path (headline)
    python bench.py --impl reference --gpus N --steps K ...        # the same workload on the CPU oracle (host cores)
    python bench.py --config c3|c4|c5|4k|rich ...                  # the other shapes, each with its own roofline
    python bench.py ... --dump-outputs DIR                         # + what the last timed step computed, as DIR/*.npy

Workloads (no real doom1.wad / doom2.wad exists in the environment: synthetic stand-ins of the same scale; set
B2D_IWAD=/path/doom1.wad to run c2 on a real one):
  c2   configs[1]  SYN_E1M1 (seed 1), 1000-pose fly-through, 1920x1080, one GPU; under torchrun every rank renders the
                   fly-through rotated by rank (weak scaling, no data-path collective)
  c3   configs[2]  nine maps E1M1-E1M9, 1000 poses each, 1920x1080, one GPU, one renderer per map, batches interleaved
  c4   configs[3]  ten maps MAP01-MAP10, 1000 poses each, 3840x2160, one map per GPU at a time (3/3/2/2 on 4 GPUs)
  c5   configs[4]  100 k random poses, 1920x1080, sharded over the ranks, chunked NCCL all-gather of finished frames
                   overlapped with rendering (b2d_render_sharded); render-only / gather-only / joint reported separately
  4k   c2 at 3840x2160 (100-pose batches);   rich: c2 on the content-rich generated level (masked middles, sprites,
                   animated / scrolling / flashing content)
One "step" is one pass of the hot path over the configuration's pose set; --steps sets how many are timed.  `value` is
device-resident throughput (poses already in HBM, frames written to HBM); `e2e` (c2) goes through b2d_render with
pinned HOST buffers -- host poses in, host frames out, both copies inside the timed region.

--dump-outputs DIR writes, after the timed steps, what the last step handed its caller (the index frames, the RGBA
frames with --rgba, c5's per-frame checksums) as float32 / float64 .npy files: a fixed, seeded sample of at most 64 MB.
Poses and levels are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "frames/sec at 1920x1080 (palette-index bit-exact)"
UNIT = "frames/s"
RICH_CFG = dict(mid_pct=30, thing_pct=40, anim=True)


# ---------------------------------------------------------------------------------------------- workloads
def workload(cfg: str, args):
    """(width, height, [(map name, wad seed, synth cfg, pose kind, pose seed)], poses per map, description)"""
    n = args.poses
    if cfg in ("c2", "4k", "rich"):
        w, h = (3840, 2160) if cfg == "4k" else (1920, 1080)
        n = n or (400 if cfg == "4k" else 1000)
        maps = [("E1M1", 1, RICH_CFG if cfg == "rich" else {}, "fly", 2)]
        what = {"c2": "configs[1]", "4k": "configs[1] at 3840x2160", "rich": "configs[1] on the content-rich level"}[cfg]
        name = "synthetic SYN_E1M1 (seed 1, E1M1-scale%s)" % (", masked middles 30 % + sprites + animated/scrolling/flashing content" if cfg == "rich" else "")
        return w, h, maps, n, "%s: %s, %d-pose fly-through per GPU, %dx%d, index framebuffer only" % (what, name, n, w, h)
    if cfg == "c3":
        n = n or 1000
        maps = [("E1M%d" % i, 10 + i, {}, "fly", 2) for i in range(1, 10)]
        return 1920, 1080, maps, n, ("configs[2]: nine synthetic maps E1M1-E1M9 (seeds 11-19), %d-pose fly-through each, "
                                     "1920x1080, one renderer per map, batches interleaved, index framebuffer only" % n)
    if cfg == "c4":
        n = n or 1000
        maps = [("MAP%02d" % i, 20 + i, {}, "fly", 2) for i in range(1, 11)]
        return 3840, 2160, maps, n, ("configs[3]: ten synthetic maps MAP01-MAP10 (seeds 21-30; doom2.wad is commercial and absent), "
                                     "%d-pose fly-through each, 3840x2160, one map per GPU at a time (3/3/2/2 on 4), no collective" % n)
    if cfg == "c5":
        n = n or 100000
        maps = [("E1M1", 1, {}, "random", 5)]
        return 1920, 1080, maps, n, ("configs[4]: synthetic SYN_E1M1 (seed 1), %d random poses (splitmix64 seed 5), 1920x1080, "
                                     "contiguous pose blocks per rank, chunked NCCL all-gather of finished index frames" % n)
    raise SystemExit("unknown --config " + cfg)


def build_wad(mapname, seed, cfg):
    from rust_doom_b200 import synthwad
    return synthwad.build_iwad(seed, (mapname,), cfg=synthwad.SynthConfig(**cfg))


def make_poses(scene, kind, n, seed):
    from rust_doom_b200 import poses as P
    return P.random_poses(scene, n, seed) if kind == "random" else P.flythrough_poses(scene, n, seed)


def bench_config(desc, n, world, scene_info, extra=None):
    """The `config` object of the JSON line: identical for this repo's arm and the reference arm."""
    c = {"workload": desc, "poses_per_step_per_gpu": n, "segs": int(scene_info.n_segs), "subsectors": int(scene_info.n_ssectors),
         "parallelism": "pose-sharded x%d" % world,
         "l2": "frames written per step >> 126 MB L2 (2.07 MB per 1080p frame); the scene (~0.3 MB) is legitimately cache-resident"}
    if extra:
        c.update(extra)
    return c


def build_provenance():
    """Which build of which sources this run measured (rust-doom_b200/libb2d.build.json, written by build())."""
    from rust_doom_b200 import _lib, build
    info = build.build_info()
    info["library"] = os.path.relpath(_lib.LIB_PATH, ROOT)
    return info


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram bytes per raster launch from the committed ncu capture (profiles/roofline.json), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline.json")) as f:
            return json.load(f).get("raster_dram_bytes_per_launch")
    except Exception:  # noqa: BLE001
        return None


DUMP_MAX_BYTES = 64 * 1000 * 1000
DUMP_SEED = 2024


def dump_share(n_outputs):
    """Bytes each of `n_outputs` outputs may take in DIR (the .npy headers fit in what is held back)."""
    return (DUMP_MAX_BYTES - (64 << 10)) // n_outputs


def sample_output(name, t, share, dtype=np.float32):
    """What --dump-outputs keeps of the output `t` (a torch tensor whose first axis is the frame) in at most `share` bytes
    of `dtype`: the whole output when it fits, else a fixed, seeded sample of it -- `<name>_values`, values at random
    positions over the whole output, so that every frame is represented, and `<name>_frames`, whole frames at random
    positions, as many as the rest of the share holds."""
    import torch

    def host(x):
        return x.cpu().numpy().astype(dtype)

    size = np.dtype(dtype).itemsize
    if t.numel() * size <= share:
        return {name: host(t)}
    rng = np.random.default_rng([DUMP_SEED, zlib.crc32(name.encode())])
    n, total = t.shape[0], t.numel()
    nval = min(total, share // size // 8)
    k = min(n, (share - nval * size) // (total // n * size))
    if k == 0:
        nval = share // size
    pos = torch.from_numpy(np.sort(rng.integers(0, total, nval))).to(t.device)
    out = {name + "_values": host(t.reshape(-1)[pos])}
    if k:
        out[name + "_frames"] = host(t[torch.from_numpy(np.sort(rng.choice(n, k, replace=False))).to(t.device)])
    return out


def write_outputs(out_dir, arrays):
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_MAX_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = sorted(sm)[len(sm) // 2:] if len(sm) > 2 else sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- CPU arm
def cpu_reference(blob, poses, width, height, threads, steps, warmup, min_seconds=0.0):
    """The oracle (the only CPU implementation of this path that exists: the reference rasterises in OpenGL) on `threads`
    host cores, OpenMP over poses.  A step renders `poses` into a buffer that is allocated -- and touched -- once, so
    that steps do not time first-touch page faults.  Returns (frames/s, ms per step, steps timed)."""
    from oracle import render
    view = render.make_view(width, height)
    out = np.zeros((len(poses), height, width), dtype=np.uint8)
    for _ in range(max(warmup, 0)):
        render.render(blob, view, poses, threads=threads, out=out)
    done = 0
    t0 = time.perf_counter()
    while True:
        render.render(blob, view, poses, threads=threads, out=out)
        done += 1
        if done >= steps and time.perf_counter() - t0 >= min_seconds:
            break
    dt = time.perf_counter() - t0
    return done * len(poses) / dt, dt / done * 1e3, done


def cpu_pose_sample(poses, cores):
    """Poses per CPU step: the whole step when the host can render it in about a second, else an evenly spaced sample."""
    cap = max(cores * 16, 64)
    if len(poses) <= cap:
        return poses, "all %d poses of the step" % len(poses)
    idx = np.linspace(0, len(poses) - 1, cap).astype(int)
    return np.ascontiguousarray(poses[idx]), "%d evenly spaced of the step's %d poses (host has %d cores)" % (cap, len(poses), cores)


def reference_arm(args, cfg):
    """`--impl reference`: the workload of --config on the host cores, through oracle/ alone (libb2d.so is not loaded)."""
    from oracle.host import OracleScene
    from rust_doom_b200.jobs import usable_cores
    width, height, maps, n, desc = workload(cfg, args)
    cores = usable_cores()
    iwad = os.environ.get("B2D_IWAD") if cfg == "c2" else None
    if iwad:
        with open(iwad, "rb") as f:
            scenes = [OracleScene(f.read(), 0)]
        desc = desc.replace("synthetic SYN_E1M1 (seed 1, E1M1-scale)",
                            "%s level 0 (%s)" % (os.path.basename(iwad), scenes[0].archive.level_name(0).rstrip(b"\0").decode()))
    else:
        scenes = [OracleScene(build_wad(m, seed, c), 0) for (m, seed, c, _, _) in maps]
    poses = [make_poses(sc, kind, n if cfg != "c5" else min(n, max(cores * 16, 64)), pseed)
             for sc, (_, _, _, kind, pseed) in zip(scenes, maps)]
    # a step = every map's sample once
    samples = [cpu_pose_sample(p, cores) for p in poses]
    from oracle import render
    view = render.make_view(width, height)
    outs = [np.zeros((len(s[0]), height, width), dtype=np.uint8) for s in samples]

    def step():
        for sc, (ps, _), out in zip(scenes, samples, outs):
            render.render(sc.blob, view, ps, threads=cores, out=out)

    for _ in range(min(max(args.warmup, 1), 2)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    frames = sum(len(s[0]) for s in samples)
    fps = args.steps * frames / dt
    sample = "%s per map x %d map(s) per step at %dx%d, OpenMP over poses, %d threads, oracle/b2d_oracle.c -O3 -march=native (%.1f frames/s per core)" % (
        samples[0][1], len(samples), width, height, cores, fps / cores)
    cb = {"value": fps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
    world = int(os.environ.get("WORLD_SIZE", "1"))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": bench_config(desc, n, world, scenes[0].info),
        "cpu_baseline": cb,
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))
    return 0


# ---------------------------------------------------------------------------------------------- checkers (oracle)
def verify_c5(b2d, jobs, result, scene, poses, width, height, rank, world, samples=8):
    """Every rank holds the same checksum for every gathered frame, and sampled frames equal the oracle's.
    (The checker: imports oracle/.)"""
    import torch
    import torch.distributed as dist
    table = result["table"]
    t = table.table
    ok_ranks = True
    if world > 1:
        lo, hi = t.clone(), t.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        ok_ranks = bool(torch.equal(lo, hi))
    host = table.host()
    per = result["per_rank"]
    n_total = len(poses)
    mism = 0
    checked = 0
    if rank == 0:
        from oracle import render as orender
        idx = np.unique(np.linspace(0, n_total - 1, samples).astype(np.int64))
        ofb = orender.render(scene.blob, orender.make_view(width, height), np.ascontiguousarray(poses[idx]), threads=jobs.usable_cores())
        for k, g in enumerate(idx):
            q, j = divmod(int(g), per)
            checked += 1
            if int(host[q, j]) != b2d.frame_checksum(ofb[k]):
                mism += 1
    return {"all_ranks_identical": ok_ranks, "oracle_samples": checked, "oracle_mismatches": mism}



def verify_maps(result, scenes, poses, width, height, probes_per_map=1):
    """One probe frame per map against the oracle (the checker: imports oracle/).  Returns mismatching frames."""
    from oracle import render as orender
    bad = 0
    view = orender.make_view(width, height)
    for m, sc in enumerate(scenes):
        n = len(poses[m])
        for k in range(probes_per_map):
            i = (n // 2 + k * 7919) % n
            ofb = orender.render(sc.blob, view, poses[m][i:i + 1], threads=1)
            if not np.array_equal(result["outs"][m][i].cpu().numpy(), ofb[0]):
                bad += 1
    return bad


# ---------------------------------------------------------------------------------------------- helpers (GPU arm)
def roofline_of(raster_ms_per_launch_set, alg_bytes, walk_ms, note, kernel="b2d_raster_kernel<index>", traffic=None):
    peak, peak_src = measured_peak()
    achieved = alg_bytes / (raster_ms_per_launch_set / 1e3) / 1e9 if raster_ms_per_launch_set > 0 else 0.0
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "kernel": kernel, "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": raster_ms_per_launch_set,
            "walk_avg_launch_ms": walk_ms, "peak_source": peak_src, "note": note}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b2d", choices=["b2d", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5", "4k", "rich"])
    ap.add_argument("--poses", type=int, default=0, help="poses per map / per job (0 = the configuration's own count)")
    ap.add_argument("--chunk", type=int, default=256, help="c5: frames per rank per all-gather chunk")
    ap.add_argument("--transports", default="ce", help="c5: comma list of exchange transports to run: ce (the library's default: copy engines "
                    "over CUDA-IPC mappings), window / register / plain (ncclAllGather on ncclMemAlloc window / registered / plain buffers)")
    ap.add_argument("--batch", type=int, default=0, help="c3/c4/4k/rich: frames per launch (0 = 500)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--no-pipeline", action="store_true",
                    help="c2: one b2d_render_device call per step (BSP walk, then raster of the same batch, one stream) instead of "
                         "the default b2d_walk_device / b2d_raster_device pair on two streams (the walk of the next batch runs as a "
                         "one-CTA-per-SM background grid under this batch's raster)")
    ap.add_argument("--raster-streams", type=int, default=2, choices=[1, 2],
                    help="pipelined step (c2) / map jobs (c3, c4, 4k, rich): 2 = consecutive batches raster on two alternating streams into two output buffers, so the "
                         "first CTAs of batch k+1 fill the SMs that the last CTAs of batch k leave idle (1 = one stream, one buffer)")
    ap.add_argument("--rgba", action="store_true", help="c2: also materialise RGBA8 frames in HBM (5 B/pixel; not the headline config)")
    ap.add_argument("--gather-frames", type=int, default=0, help="c2, N>1: frames per rank in a separate all-gather timing (0 = off; see --config c5)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed (rank 0's "
                    "outputs) as DIR/<name>.npy: float32 (float64 for c5's checksums), a fixed, seeded sample of at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b2d)")
    args.warmup = max(args.warmup, 0)
    cfg = args.config
    # stdout carries the one JSON line: NCCL's version banner / debug output (NCCL_DEBUG may be set by the box) goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        return reference_arm(args, cfg)

    import torch
    import torch.distributed as dist

    import rust_doom_b200 as b2d
    from rust_doom_b200 import jobs

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = {"bound": False} if args.no_numa else jobs.bind_to_gpu_numa(local_rank)   # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cores = jobs.usable_cores()
    args.warmup = max(args.warmup, 3)          # timing hygiene: at least 3 warm-up steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    width, height, maps, n, desc = workload(cfg, args)
    npix = width * height

    # ================================================================== c5: sharded render + overlapped all-gather
    if cfg == "c5":
        mapname, seed, scfg, kind, pseed = maps[0]
        scene = b2d.Scene(b2d.Archive.from_bytes(build_wad(mapname, seed, scfg)), 0)
        poses = make_poses(scene, kind, n, pseed)                     # identical on every rank (deterministic)
        # exchange transports to try (best joint throughput is reported as the line's value, all of them under "transports"):
        #   window  ncclAllGather in place on ncclMemAlloc buffers registered as a symmetric window (NCCL >= 2.27)
        #   plain   ncclAllGather in place on cudaMalloc buffers, no registration
        #   ce      copy engines: every rank pushes its slice into the peers' buffers over CUDA-IPC mappings
        env_of = {"window": {"B2D_GATHER": "nccl"}, "register": {"B2D_GATHER": "nccl", "B2D_NCCL_NO_WINDOW": "1"},
                  "plain": {"B2D_GATHER": "nccl", "B2D_NCCL_NO_REGISTER": "1"}, "ce": {}}
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        results, checksums = {}, {}
        for tname in [t for t in args.transports.split(",") if t]:
            for k in ("B2D_NCCL_NO_WINDOW", "B2D_NCCL_NO_REGISTER", "B2D_GATHER"):
                os.environ.pop(k, None)
            os.environ.update(env_of[tname])
            comm = jobs.make_comm(local_rank) if world > 1 else jobs.single_comm(local_rank)
            r1 = jobs.run_c5(scene, poses, width, height, local_rank, comm, chunk=args.chunk, reps=args.steps)
            v1 = verify_c5(b2d, jobs, r1, scene, poses, width, height, rank, world)
            if not v1["all_ranks_identical"] or v1["oracle_mismatches"] or r1["status_bits"]:
                raise SystemExit("c5 validation failed (%s): %r status %d" % (tname, v1, r1["status_bits"]))
            table = r1.pop("table")
            r1.pop("renderer")
            if args.dump_outputs and rank == 0:
                checksums[tname] = table.host()
            results[tname] = (r1, v1)
            comm.close()
            torch.cuda.empty_cache()
        clocks = sampler.stop() if rank == 0 else None
        best = max(results, key=lambda t: results[t][0]["joint_fps"])
        res, ver = results[best]
        keys = ("n_total", "frames", "per_rank", "chunk_frames", "chunks", "render_only_ms", "gather_only_ms", "joint_ms", "joint_checked_ms",
                "render_only_fps", "gather_only_fps", "joint_fps", "joint_checked_fps", "gather_gbs_received_per_rank",
                "joint_gbs_received_per_rank", "registration", "nccl_version")
        if rank == 0:
            if args.dump_outputs:       # per-frame checksums of every gathered frame, [rank, frame of the rank's slice]
                write_outputs(args.dump_outputs, sample_output("checksums", torch.from_numpy(checksums[best].astype(np.int64)),
                                                               dump_share(1), np.float64))
            nvl = 900.0
            print(json.dumps({
                "metric": METRIC, "value": res["joint_fps"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": 1,
                "ms_per_step": res["joint_ms"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic",
                "config": bench_config(desc, res["per_rank"], world, scene.info,
                                       {"chunk_frames_per_rank": res["chunk_frames"], "chunks": res["chunks"], "transport": best,
                                        "step": "the whole job: render + all-gather of every chunk, overlapped (b2d_render_sharded); "
                                                "`value` = joint frames/s, NVLink-bound"}),
                "clocks": clocks, "gpu_launches": int(2 * res["chunks"] * 4),
                "c5": {k: res[k] for k in keys},
                "transports": {t: {k: results[t][0][k] for k in keys} for t in results},
                "c5_bounds": {"nvlink_gbs_per_direction": nvl,
                              "gather_frac_of_nvlink": res["gather_gbs_received_per_rank"] / nvl if world > 1 else None,
                              "joint_over_gather_only": res["joint_fps"] / res["gather_only_fps"] if res["gather_only_fps"] else None},
                "validation": ver,
                "roofline": {"bound": "nvlink", "achieved": res["joint_gbs_received_per_rank"], "peak": nvl, "unit": "GB/s",
                             "frac": res["joint_gbs_received_per_rank"] / nvl if world > 1 else None, "traffic": None,
                             "note": "bytes received per rank per second in the joint run vs one NVLink-5 direction (SURVEY.md 0.5); "
                                     "render-only throughput is the HBM-bound number of --config c2"}}))
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ================================================================== c3 / c4 / 4k / rich: several maps or other shapes
    if cfg in ("c3", "c4", "4k", "rich"):
        mine = jobs.map_assignment(len(maps), world)[rank] if cfg == "c4" else list(range(len(maps)))
        # frames per launch: the BSP walk is one latency-bound wave (~0.1 ms whatever the batch), so batches are large;
        # c3 still interleaves the nine renderers batch by batch
        batch = args.batch or min(n, 500)
        scenes, poses = [], []
        for m in mine:
            mapname, seed, scfg, kind, pseed = maps[m]
            sc = b2d.Scene(b2d.Archive.from_bytes(build_wad(mapname, seed, scfg)), 0)
            scenes.append(sc)
            ps = make_poses(sc, kind, n, pseed)
            poses.append(np.roll(ps, -(rank * n // max(world, 1))) if cfg != "c4" else ps)
        steps = args.steps
        dump = args.dump_outputs and rank == 0
        dumped = {}
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        barrier()
        if cfg == "c4" and len(scenes) > 1:
            # one map at a time (frames of a 4K map: 8.3 GB per 1000): keep one output buffer alive
            tot = {"ms_per_pass": 0.0, "raster_ms_per_pass": 0.0, "walk_ms_per_pass": 0.0, "frames_per_pass": 0, "launches": 0, "status_bits": 0}
            bad = 0
            for m, sc, ps in zip(mine, scenes, poses):
                r1 = jobs.run_maps([sc], [ps], width, height, local_rank, batch, steps, args.warmup, False, args.raster_streams)
                bad += verify_maps(r1, [sc], [ps], width, height)
                if dump:
                    dumped.update(sample_output(maps[m][0] + "_index", r1["outs"][0], dump_share(len(scenes))))
                for k in tot:
                    tot[k] += r1[k]
                del r1
                torch.cuda.empty_cache()
            res = tot
        else:
            res = jobs.run_maps(scenes, poses, width, height, local_rank, batch, steps, args.warmup, cfg == "c3", args.raster_streams)
            bad = verify_maps(res, scenes, poses, width, height)
            if dump:
                for m, out in zip(mine, res["outs"]):
                    dumped.update(sample_output(maps[m][0] + "_index", out, dump_share(len(scenes))))
        if dump:
            write_outputs(args.dump_outputs, dumped)
        clocks = sampler.stop() if rank == 0 else None
        if bad or res["status_bits"]:
            raise SystemExit("parity check failed: %d probe frame(s) differ from the oracle, status %d" % (bad, res["status_bits"]))
        ms = max_over_ranks(res["ms_per_pass"])
        frames = torch.tensor([res["frames_per_pass"]], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(frames)
        total_frames = float(frames.item())
        value = total_frames / (ms / 1e3)
        roof = roofline_of(res["raster_ms_per_pass"], float(res["frames_per_pass"]) * npix, res["walk_ms_per_pass"],
                           "this rank's raster launches of one pass vs the index bytes they write; index-only output" +
                           ("; the launches alternate between two streams and overlap by their tails, with the next launch's BSP walk "
                            "co-resident: their time is the pass" if args.raster_streams > 1 else " (sum of the per-launch event pairs)"))
        if rank == 0:
            print(json.dumps({
                "metric": METRIC if height == 1080 else METRIC.replace("1920x1080", "%dx%d" % (width, height)),
                "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if cfg == "c4" else "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic",
                "config": bench_config(desc, n, world, scenes[0].info,
                                       {"maps_this_rank": len(scenes), "batch": batch,
                                        "raster_streams": res.get("raster_streams", args.raster_streams),
                                        "step": "one pass over every map of the rank (%s)" % ("batches interleaved across the maps' renderers" if cfg == "c3" else "map after map")}),
                "clocks": clocks, "gpu_launches": int(res["launches"]), "roofline": roof,
                "parity": "one probe frame per map bit-exact vs the oracle"}))
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ================================================================== c2: the headline configuration
    iwad = os.environ.get("B2D_IWAD")
    if iwad:
        arch = b2d.Archive.open(iwad)
        desc = desc.replace("synthetic SYN_E1M1 (seed 1, E1M1-scale)", "%s level 0 (%s)" % (os.path.basename(iwad), arch.level_name(0)))
    else:
        arch = b2d.Archive.from_bytes(build_wad(*maps[0][:3]))
    scene = b2d.Scene(arch, 0)
    # every rank renders the same fly-through, cyclically rotated by rank: identical work per GPU (clean weak-scaling
    # efficiency) while no two ranks are on the same pose at the same time
    poses_np = np.roll(make_poses(scene, "fly", n, 2), -(rank * n // max(world, 1)))
    view = b2d.make_view(width, height)
    r = b2d.Renderer(scene, view, device=local_rank, max_batch=n)
    d_poses = torch.from_numpy(poses_np.view(np.int32).reshape(-1, 4).copy()).to(dev)
    pipelined = not args.no_pipeline
    masked = scene.info.n_masked_mids + scene.info.n_sprites > 0      # such rasters are ordered by an event: one stream
    nbuf = args.raster_streams if pipelined and not masked else 1
    d_index_all = [torch.empty((n, height, width), dtype=torch.uint8, device=dev) for _ in range(nbuf)]
    d_rgba_all = [torch.empty((n, height, width), dtype=torch.int32, device=dev) if args.rgba else None for _ in range(nbuf)]
    d_index, d_rgba = d_index_all[0], d_rgba_all[0]
    main_stream = torch.cuda.current_stream()
    stream = main_stream.cuda_stream

    walk_stream = torch.cuda.Stream(device=dev, priority=-1) if pipelined else None
    raster_streams = [torch.cuda.Stream(device=dev) for _ in range(nbuf)] if pipelined and nbuf > 1 else None
    pending = [r.walk_device(d_poses.data_ptr(), n, walk_stream.cuda_stream)] if pipelined else None
    turn = [0]

    def step():
        if pipelined:
            b = turn[0] % nbuf
            turn[0] += 1
            rs = raster_streams[b].cuda_stream if raster_streams else stream
            r.raster_device(pending[0], d_index_all[b].data_ptr(), d_rgba_all[b].data_ptr() if args.rgba else 0, rs)
            pending[0] = r.walk_device(d_poses.data_ptr(), n, walk_stream.cuda_stream)
        else:
            r.render_device(d_poses.data_ptr(), n, d_index.data_ptr(), d_rgba.data_ptr() if args.rgba else 0, stream)

    def join():                                 # the main stream waits for everything the steps enqueued elsewhere
        if raster_streams:
            for t in raster_streams:
                main_stream.wait_stream(t)

    def fork():                                 # ... and the side streams start behind the main stream
        if raster_streams:
            for t in raster_streams:
                t.wait_stream(main_stream)

    fork()
    for _ in range(max(args.warmup, nbuf)):
        step()
    join()
    barrier()
    # parity spot check inside the run: one frame of this batch (of every output buffer) against the oracle rendering the
    # scene its own loader and compiler produce from the same WAD bytes
    if rank == 0:
        from oracle import render as orender, scene as oscene, wad as owad
        oarch = owad.Archive(open(iwad, "rb").read() if iwad else build_wad(*maps[0][:3]))
        oblob = oscene.compile_scene(oarch, owad.TextureDirectory(oarch), 0)
        probe = n // 2
        ofb = orender.render(oblob, orender.make_view(width, height), poses_np[probe:probe + 1])
        for buf in d_index_all:
            if not np.array_equal(buf[probe].cpu().numpy(), ofb[0]):
                raise SystemExit("parity check failed: GPU frame differs from the oracle")

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = r.launch_count
    r.profile(True)
    r.profile_read()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fork()
    for _ in range(args.steps):
        step()
    join()
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:        # the buffers the last step rastered into, before anything else writes them
        b = (turn[0] - 1) % nbuf if pipelined else 0
        outs = {"index": d_index_all[b]}
        if args.rgba:                          # RGBA8 per pixel, as channels
            outs["rgba"] = d_rgba_all[b].view(torch.uint8).reshape(n, height, width, 4)
        dumped = {}
        for name, t in outs.items():
            dumped.update(sample_output(name, t, dump_share(len(outs))))
        write_outputs(args.dump_outputs, dumped)
    if pipelined:                              # the walk issued by the last step belongs to a step that never comes
        r.raster_device(pending[0], d_index.data_ptr(), d_rgba.data_ptr() if args.rgba else 0, stream)
        torch.cuda.synchronize()
    ms_total = e0.elapsed_time(e1)
    walk_ms, raster_ms, batches = r.profile_read()
    r.profile(False)
    launches = r.launch_count - launches0
    clocks = sampler.stop() if rank == 0 else None
    status = r.status()                        # sticky completeness bits of the device-resident path
    if status:
        raise SystemExit("renderer status %d: frames incomplete" % status)
    ms_total = max_over_ranks(ms_total)
    value = world * n * args.steps / (ms_total / 1e3)

    alg_bytes = float(n) * npix * (5 if args.rgba else 1)
    overlapped = raster_streams is not None
    # rasters of consecutive batches on alternating streams overlap (head of k+1 in the tail of k), so an event pair around
    # one launch also spans its wait for SMs: the kernel's duration in the timed region is then the region over its launches
    per_launch = ms_total / args.steps if overlapped else raster_ms / max(batches, 1)
    roofline = roofline_of(per_launch, alg_bytes, walk_ms / max(batches, 1),
                           "index-only output (no RGBA materialised); the raster kernel is instruction-issue / L1 bound, not HBM bound "
                           "(DESIGN.md 5-6, profiles/README.md)" +
                           ("; avg_launch_ms = timed region / raster launches: the rasters run back to back on two streams, overlapping by "
                            "their tails, with the next batch's BSP walk co-resident" if overlapped else ""),
                           "b2d_raster_kernel<%s>" % ("rgba" if args.rgba else "index"), None if args.rgba else ncu_traffic())
    if pipelined:        # the same kernel timed alone, outside the timed region: one stream, walk first, nothing co-resident
        r.profile(True)
        r.profile_read()
        for _ in range(10):
            r.render_device(d_poses.data_ptr(), n, d_index.data_ptr(), d_rgba.data_ptr() if args.rgba else 0, stream)
        torch.cuda.synchronize()
        _, alone_ms, alone_n = r.profile_read()
        r.profile(False)
        alone = max_over_ranks(alone_ms / max(alone_n, 1))
        roofline["alone_avg_launch_ms"] = alone
        roofline["alone_frac"] = alg_bytes / (alone / 1e3) / 1e9 / roofline["peak"]

    # ------------------------------------------------------------------ end to end (host buffers)
    e2e = None
    if not args.no_e2e:
        e2e_n = n
        r2 = b2d.Renderer(scene, view, device=local_rank, max_batch=min(125, e2e_n))
        h_poses = torch.from_numpy(poses_np.view(np.int32).reshape(-1, 4).copy()).pin_memory()
        h_index = torch.empty((e2e_n, height, width), dtype=torch.uint8).pin_memory()
        r2.render_ptr(h_poses.data_ptr(), e2e_n, h_index.data_ptr())        # warm-up (allocations)
        e2e_steps = max(1, min(args.steps, 3))
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            r2.render_ptr(h_poses.data_ptr(), e2e_n, h_index.data_ptr())
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": world * e2e_n * e2e_steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(poses_np.nbytes), "d2h_bytes_per_step": int(e2e_n * npix),
               "steps": e2e_steps, "d2h_gbs_per_gpu": e2e_n * e2e_steps * npix / dt / 1e9,
               "api": "b2d_render (pinned host poses in, pinned host frames out, double-buffered D2H on two copy streams)",
               "numa": numa,
               "note": "PCIe-bound: one 1080p index frame is 2.07 MB over a ~57 GB/s Gen5 x16 link = ~27.5 k frames/s per GPU"}
        if rank == 0 and not np.array_equal(h_index[n // 2].numpy(), d_index[n // 2].cpu().numpy()):
            raise SystemExit("e2e path disagrees with the device path")
        del r2

    # ------------------------------------------------------------------ optional frame all-gather (N>1), separate
    allgather = None
    if world > 1 and args.gather_frames > 0:
        comm = jobs.make_comm(local_rank)
        g = min(args.gather_frames, n)
        st = r.render_sharded(comm, np.tile(poses_np[:g], world), g, b2d._lib.SHARD_GATHER_ONLY)
        st = r.render_sharded(comm, np.tile(poses_np[:g], world), g, b2d._lib.SHARD_GATHER_ONLY)
        gms = max_over_ranks(st["total_ms"])
        allgather = {"frames": g * world, "ms": gms, "frames_per_s": g * world / (gms / 1e3),
                     "note": "in-place NCCL all-gather of finished index frames (b2d_render_sharded, gather only), NVLink-bound, NOT part of `value`; the full job is --config c5"}
        comm.close()

    # ------------------------------------------------------------------ CPU baseline (rank 0, N=1 only)
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ps, what = cpu_pose_sample(poses_np, cores)
        fps, ms, done = cpu_reference(scene.blob, ps, width, height, cores, 1, 1, min_seconds=8.0)
        cpu_baseline = {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": "%s x %d passes at %dx%d, OpenMP over poses, %d threads, oracle/b2d_oracle.c -O3 -march=native (%.1f frames/s per core)"
                                  % (what, done, width, height, cores, fps / cores)}

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": bench_config(desc + (", + RGBA8 framebuffer" if args.rgba else ""), n, world, scene.info),
            "step": ("raster of this batch + BSP walk of the NEXT batch (b2d_walk_device / b2d_raster_device): every step runs one walk "
                     "and one raster of 1000 poses, the walk as a background grid under the raster" +
                     ("; rasters alternate between two streams and two output buffers (the first CTAs of batch k+1 use the SMs the "
                      "last CTAs of batch k leave idle)" if overlapped else "; roofline.avg_launch_ms is the raster's duration WITH that walk co-resident")
                     if pipelined else "BSP walk then raster of one batch, one stream (b2d_render_device)"),
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
            "cpu_baseline": cpu_baseline, "allgather": allgather, "build": build_provenance()}))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
