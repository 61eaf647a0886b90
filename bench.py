#!/usr/bin/env python3
"""bench.py — env-steps/s of the batched Simulator.step() hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--envs E] [--map M] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path over one batch: `env.step(actions)` for all E envs of the
rank (pose integration, lane/reward/collision, 160x120 render, device-side auto-reset).  Workload
at every N: BASELINE.json configs[1] per GPU (Duckietown-small_loop stand-in, 4096 envs, 160x120,
uniform random [vel, steer] actions, domain_rand off) -> weak scaling.  Prints ONE JSON line.
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
sys.path.insert(0, ROOT)

METRIC = "env-steps/sec (obs+reward+done) at N envs, 1/2/4/8 B200 vs CPU ref"
UNIT = "env-steps/s"


def usable_cores():
    """Host cores this process may actually use: affinity mask and cgroup CPU quota, not os.cpu_count()."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


def b_alg(w, h):
    """Algorithmic bytes per env-step (SURVEY 8d): obs store + bilinear RGBA8 texel reads + state."""
    return w * h * (3 + 16) + 256


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.q = ("index,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                  "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                  "clocks_event_reasons.sw_power_cap")
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([c.strip() for c in line.split(",")])
            except Exception:
                pass
            time.sleep(0.15)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def cpu_reference_run(map_name, w, h, steps, warmup, sample_envs, threads):
    """The CPU arm: oracle port of Simulator.step() (logic + software render), one env per OpenMP
    task on all host cores.  Returns (env_steps_per_s, seconds, description)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as orc
    from gym_duckietown_b200 import maps

    md = maps.load_map(map_name)
    rng = np.random.default_rng(1234)
    tiles = [md.drivable_tiles[k % len(md.drivable_tiles)] for k in range(sample_envs)]
    # spawn on lane centres of drivable tiles (valid poses), like a reset would
    px = np.array([(i + 0.5) * md.tile_size for i, j in tiles]) + 0.0
    pz = np.array([(j + 0.5) * md.tile_size for i, j in tiles]) + 0.0
    om = orc.OracleMap(md)
    ang = np.zeros(sample_envs)
    for k in range(sample_envs):  # pick a heading that is a valid spawn
        for a in np.linspace(-np.pi, np.pi, 16, endpoint=False):
            o = om.done_reward(px[k], pz[k], a, 0)
            if not o.done and o.in_lane and abs(o.lane_angle) < 0.5:
                ang[k] = a
                break
    batch = orc.OracleBatch(md, px, pz, ang, W=w, H=h, threads=threads)
    acts = rng.uniform(-1, 1, (warmup + steps, sample_envs, 2)).astype(np.float32)
    # shared hosts often expose more logical CPUs than they let one tenant run: pick the thread count
    # that is actually fastest (2 trial steps each) so the CPU arm is not handicapped by oversubscription
    best = (0.0, threads)
    for cand in sorted({threads, max(1, threads // 2), max(1, threads // 4), min(threads, 32), min(threads, 16)}):
        batch.threads = cand
        batch.step(acts[0])
        t0 = time.perf_counter()
        batch.step(acts[0]); batch.step(acts[1])
        rate = 2 * sample_envs / (time.perf_counter() - t0)
        if rate > best[0]:
            best = (rate, cand)
    threads = batch.threads = best[1]
    for t in range(warmup):
        batch.step(acts[t])
    t0 = time.perf_counter()
    for t in range(steps):
        batch.step(acts[warmup + t])
    dt = time.perf_counter() - t0
    return sample_envs * steps / dt, dt, threads, (f"{sample_envs} envs x {steps} steps of the same workload "
                                                   f"(oracle port: C logic + software rasteriser, {threads} OpenMP threads)")


BASELINE_CONFIGS = {
    # BASELINE.json configs[1..4] (configs[0] is the reference's own 1-env CPU case = the --impl reference arm)
    "c2": dict(map="small_loop", envs=4096, width=160, height=120, domain_rand=False, distortion=False, cycle=False),
    "c3": dict(map="loop_obstacles", envs=4096, width=160, height=120, domain_rand=False, distortion=False, cycle=False),
    "c4": dict(map="udem1", envs=8192, width=640, height=480, domain_rand=True, distortion=True, cycle=False),
    "c5": dict(map="small_loop,loop_obstacles,udem1,loop_pedestrians,loop_dyn_duckiebots,loop_trafficlights",
               envs=4096, width=160, height=120, domain_rand=False, distortion=False, cycle=True),
    # c2 with the LITERAL road tiles of simulator.py:386-507 (98 lit triangles per tile, DTS_FLAG_TESSELLATE = spec tile
    # mode 0) instead of the analytic quad + lattice the headline uses (tile mode 1): the price of the literal reading
    "c2_literal": dict(map="small_loop", envs=4096, width=160, height=120, domain_rand=False, distortion=False, cycle=False,
                       tessellate=True),
}
PARITY_UNPINNED = ["dynamics (duckietown_world DB18 model restated, source absent)",
                   "pixels (no OpenGL here: raster spec of DESIGN.md 5; render INPUTS pinned by tests/golden/gltrace_*.npz)"]


def workload_text(c):
    return (f"Duckietown-{c['map']}-v0 (stand-in map{'s, cycled on reset (MultiMap)' if c['cycle'] else ''}"
            f"{'; road tiles as the literal 98 triangles (tile mode 0)' if c.get('tessellate') else ''}), {c['envs']} envs/GPU, "
            f"{c['width']}x{c['height']} RGB, random [vel,steer] actions, domain_rand={c['domain_rand']}, "
            f"distortion={c['distortion']}, device-side auto-reset")


DUMP_BYTES = 60_000_000   # below 64 MB in all, .npy headers included


def dump_outputs(out_dir, obs, reward, done, info):
    """Write what env.step() handed its caller -- obs, reward, done and every per-env array of info -- to
    out_dir/<name>.npy: uint8 / bool / float32 as float32, wider types as float64, values unchanged.  When all envs do
    not fit DUMP_BYTES, a fixed seeded sample of them is written and env_index.npy names the envs kept, so two builds
    run with the same arguments can be compared array for array."""
    import torch
    arrays = {"obs": obs, "reward": reward, "done": done, **{f"info_{k}": v for k, v in info.items()}}
    narrow = (torch.uint8, torch.bool, torch.float32)
    per_env = 8 + sum(t[0].numel() * (4 if t.dtype in narrow else 8) for t in arrays.values())
    E = obs.shape[0]
    n = min(E, DUMP_BYTES // per_env)
    idx = np.arange(E) if n == E else np.sort(np.random.default_rng(0).choice(E, n, replace=False))
    sel = torch.from_numpy(idx).to(obs.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "env_index.npy"), idx.astype(np.float64))
    for name, t in arrays.items():
        t = t.index_select(0, sel).to(torch.float32 if t.dtype in narrow else torch.float64)
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy())


def run_config(c, K, Wm, rank, world, local_rank, obs_format="hwc_uint8", sampler=None, gather=True, gather_impl="fused",
               dump_dir=None):
    """Device-resident arm of one workload: W warm-up steps, K timed steps (k_step_logic + render) bracketed by
    barrier + synchronize, + the end-of-rollout NCCL all-gather when world > 1.  With dump_dir, the outputs of the
    last timed step are written there (dump_outputs).  Returns (result dict, env) — the env is left alive for the
    caller's end-to-end arm."""
    import torch
    import torch.distributed as dist
    from gym_duckietown_b200.batched_env import BatchedDuckietownEnv

    dev = torch.device("cuda", local_rank)
    E, W, H = c["envs"], c["width"], c["height"]
    names = c["map"].split(",")
    env = BatchedDuckietownEnv(E, names if len(names) > 1 else names[0], device=local_rank, camera_width=W, camera_height=H,
                               domain_rand=c["domain_rand"], distortion=c["distortion"], cycle_maps=c["cycle"],
                               seed=1000, auto_reset=True, device_reset=True, env_id_offset=rank * E,
                               tessellate_tiles=bool(c.get("tessellate", False)))
    if obs_format != "hwc_uint8":
        lay, dt = obs_format.split("_")
        env.set_output_format(obs_layout=lay, obs_dtype=dt)
    env.reset()
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    actions = torch.rand((K + Wm, E, 2), device=dev, generator=gen) * 2 - 1   # Box(-1,1,(2,)).sample() distribution
    gathered = ag = fg = None
    gather_note = None
    if world > 1 and gather:
        if gather_impl == "fused":
            try:   # the exchange fused into the last step's rasteriser: peer-memory stores over NVLink (dts_gather_*)
                from gym_duckietown_b200.dist import FusedObsGather
                fg = FusedObsGather(env, rank, world)
                gather_note = "fused: last step's k_raster stores every frame into all ranks' gather buffers (cudaIpc peer memory over NVLink)"
            except Exception as ex:
                gather_note = f"fused gather unavailable ({type(ex).__name__}: {ex}); NCCL all-gather"
        ok = torch.tensor([1 if fg is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)   # every rank must have mapped every peer, else all fall back
        if int(ok.item()) == 0:
            fg = None
        if fg is None:
            from gym_duckietown_b200.dist import ObsAllGather
            ag = ObsAllGather(env, rank, world)
            gathered = torch.empty((world,) + tuple(env.obs.shape), dtype=env.obs.dtype, device=dev)
            gather_note = gather_note or "NCCL all-gather after the last step (dts_allgather_obs)"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for t in range(Wm):
        if fg is not None and t == Wm - 1:
            fg.arm()              # first peer stores map the pages: keep that out of the timed region
        env.step(actions[t])
    if fg is not None:
        fg.finish()
    if ag is not None:
        ag.all_gather(gathered)   # first collective on a communicator sets up channels: keep it out of the timed region
    barrier()
    if sampler is not None:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = env.launch_count()
    env.sim.profile(1)        # two CUDA events per step around k_raster, on the launching stream (roofline)
    ev0.record()
    for t in range(K):
        if fg is not None and t == K - 1:
            fg.arm()                              # the rollout's last step also fills every rank's gather buffer
        out = env.step(actions[Wm + t])           # dts_step: k_step_logic (+ device auto-reset) + the render kernels
    if ag is not None:
        ag.all_gather(gathered)                   # baseline: the single end-of-rollout NCCL all-gather (SURVEY 8e)
    ev1.record()
    barrier()
    if dump_dir is not None:
        dump_outputs(dump_dir, *out)              # before the untimed steps below overwrite obs and state
    env.sim.profile(0)
    launches = env.launch_count() - launches0
    env.check()   # no frame hit a capacity limit
    raster_ms_sum, raster_frames = env.sim.profile_read()
    # per-kernel breakdown: a few extra (untimed) steps with an event at every kernel boundary
    env.sim.profile(2)
    for t in range(min(K, 8)):
        env.step(actions[Wm + t])
    env.sim.profile(0)
    try:
        n_cells = env.maps[0].grid_w * env.maps[0].grid_h
        pairs_per_env = env.sim.debug_frame(0, n_cells)["batch_pairs"] / E if not env.cfg.flags & 16 else None
    except Exception:
        pairs_per_env = None
    ms = ev0.elapsed_time(ev1)
    kms, frames = env.sim.profile_read()
    if world > 1:
        tmax = torch.tensor([ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax.item())
    value = world * E * K / (ms / 1000.0)
    per = {k: v / max(frames, 1) for k, v in kms.items()}
    peak, peak_src = measured_peak()
    raster_ms = raster_ms_sum["k_raster"] / max(raster_frames, 1)   # mean over the K timed steps
    achieved = E * b_alg(W, H) / (raster_ms / 1000.0) / 1e9
    render_ms = sum(per.values())
    res = {
        "value": value, "unit": UNIT, "ms_per_step": ms / K, "steps": K, "warmup": Wm, "gpu_launches": int(launches),
        "workload": workload_text(c), "gather": gather_note,
        "roofline": {"bound": "hbm", "kernel": "k_raster (dominant kernel of the step; CUDA events on the launching stream, mean over the timed steps)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": E * b_alg(W, H), "kernel_ms": raster_ms,
                     "compulsory_frac": (E * (W * H * 3 + 256) / (raster_ms / 1000.0) / 1e9) / peak,
                     "all_render_kernels_ms": render_ms, "frac_all_render_kernels": (E * b_alg(W, H) / (render_ms / 1000.0) / 1e9) / peak},
        "kernel_ms": per, "pairs_per_env": pairs_per_env,
    }
    return res, env


def bind_numa(local_rank):
    try:
        from gym_duckietown_b200.dist import bind_to_gpu_numa
        return bind_to_gpu_numa(local_rank)
    except Exception as e:   # affinity is an optimisation, never a reason to fail the bench
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="dtsim", choices=["dtsim", "reference"])
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--map", default="small_loop")
    ap.add_argument("--width", type=int, default=160)
    ap.add_argument("--height", type=int, default=120)
    ap.add_argument("--cpu-sample-envs", type=int, default=1024)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--domain-rand", action="store_true", help="BASELINE config 4: domain randomization on")
    ap.add_argument("--distortion", action="store_true", help="BASELINE config 4: fused fisheye gather")
    ap.add_argument("--obs-format", default="hwc_uint8",
                    help="fused wrapper output (SURVEY 8f-3): <hwc|chw|cwh>_<uint8|float32>; default is render_obs's own")
    ap.add_argument("--pipeline-depth", type=int, default=2, help="HostPipeline slots in flight for the e2e arm")
    ap.add_argument("--cycle-maps", action="store_true", help="BASELINE config 5: --map a,b cycled on reset (MultiMap)")
    ap.add_argument("--configs", default="auto",
                    help="extra BASELINE configs timed after the headline and attached as \"configs\": comma list of "
                         "c3,c4,c5, 'none', or 'auto' (N=1: c3,c4,c5; N>1: c5 with the NCCL all-gather)")
    ap.add_argument("--c4-envs", type=int, default=8192)
    ap.add_argument("--gather", default="fused", choices=["fused", "nccl"],
                    help="N>1: end-of-rollout observation exchange fused into the last step's rasteriser (peer memory), or NCCL")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write obs / reward / done / info of the headline's last timed step (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    W, H, E = args.width, args.height, args.envs
    cores = usable_cores()
    head = dict(map=args.map, envs=E, width=W, height=H, domain_rand=args.domain_rand, distortion=args.distortion,
                cycle=args.cycle_maps)
    config = {"workload": workload_text(head), "envs_per_gpu": E, "width": W, "height": H, "map": args.map,
              "tile_mode": "1 (one quad per road tile + analytic 8x8 lattice lighting); vs mode 0 (the literal 98 triangles, DTS_FLAG_TESSELLATE): > 1 LSB on < 1 % of the channel values, all at tile outlines (tests/test_oracle_raster.py)",
              "l2": "obs batch written per step (%.0f MB) exceeds the 126 MB L2; no flush needed" % (E * W * H * 3 / 1e6)}

    if args.impl == "reference":
        # The reference's own Pyglet/OpenGL path cannot run in this image (no pyglet, GL, display,
        # duckietown_world); the CPU arm is the oracle port of the same step on all host cores.
        if rank != 0:
            return
        k, w_ = max(1, args.steps), max(0, args.warmup)   # the driver's step / warm-up counts, as given
        val, secs, cores, desc = cpu_reference_run(args.map.split(",")[0], W, H, k, w_, args.cpu_sample_envs, cores)
        line = {"metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": k, "warmup": w_,
                "ms_per_step": 1000 * secs / k, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64 logic / f32 raster / u8 obs", "data": "synthetic", "config": config, "impl": "reference",
                "baseline_is": "C port of the reference's CPU path (oracle/), NOT the Pyglet reference itself (cannot run here)",
                "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc},
                "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    numa = bind_numa(local_rank)   # before any pinned allocation: host buffers land on the GPU's NUMA node
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    K, Wm = args.steps, max(3, args.warmup)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm: `value` -------------------------------------------------------------
    sampler = ClockSampler(local_rank) if rank == 0 else None
    res, env = run_config(head, K, Wm, rank, world, local_rank, args.obs_format, sampler, gather_impl=args.gather,
                          dump_dir=args.dump_outputs if rank == 0 else None)
    config["gather"] = res.get("gather")
    if args.obs_format != "hwc_uint8":
        config["obs_format"] = args.obs_format

    # ---- end-to-end arm: host buffers in/out through the public API -----------------------------------
    # HostPipeline.submit(): pinned-host actions -> device, dts_step, obs/reward/done -> pinned host on a copy
    # stream; result(): wait for that step's host buffers.  Two slots in flight, so the D2H of step k overlaps
    # the kernels of step k+1 (random-action rollout: actions do not depend on observations).
    from collections import deque
    from gym_duckietown_b200.batched_env import HostPipeline

    def e2e_arm(env, Ke):
        h_act = torch.empty((Ke + 3, env.num_envs, 2), dtype=torch.float32).uniform_(-1, 1).pin_memory()
        pipe = HostPipeline(env, depth=args.pipeline_depth)
        for t in range(3):
            pipe.result(pipe.submit(h_act[t]))
        barrier()
        t0 = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pend = deque()
        checksum = 0

        def consume(tk):
            ho, hr, hd = pipe.result(tk)
            return int(ho.reshape(-1)[0]) + int(hd[0])       # the host really reads the step's result

        for t in range(Ke):
            pend.append(pipe.submit(h_act[3 + t]))
            if len(pend) >= args.pipeline_depth:
                checksum += consume(pend.popleft())
        while pend:
            checksum += consume(pend.popleft())
        e1.record()
        barrier()
        ems = max(e0.elapsed_time(e1), 1000.0 * (time.perf_counter() - t0))   # device and wall clock agree; take the larger
        if world > 1:
            tmax = torch.tensor([ems], device=dev)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            ems = float(tmax.item())
        out_bytes = int(pipe.slots[0]["h_obs"].numel() * pipe.slots[0]["h_obs"].element_size())
        return {"value": world * env.num_envs * Ke / (ems / 1000.0), "unit": UNIT, "h2d_bytes_per_step": env.num_envs * 2 * 4,
                "d2h_bytes_per_step": out_bytes + env.num_envs * (4 + 1), "steps": Ke,
                "api": f"HostPipeline.submit/result, depth {args.pipeline_depth} (D2H of step k overlaps step k+1)"}

    Ke = max(5, min(K, 50))
    e2e = e2e_arm(env, Ke)
    e2e_resized = None
    if hasattr(env, "set_resize"):   # fused ResizeWrapper (wrappers.py:111-141): the training stack's 84x84 payload
        try:
            env.set_resize(84, 84)
            e2e_resized = e2e_arm(env, Ke)
            e2e_resized["obs"] = "84x84 RGB resized on the device (cv2.INTER_CUBIC semantics of ResizeWrapper)"
            env.set_resize(None, None)
        except Exception as ex:
            e2e_resized = {"error": str(ex)}
    if sampler is not None:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    env.close()
    del env
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, same step count, device-resident ---------------------------------
    extra = {}
    want = args.configs
    if want == "auto":
        want = "c3,c4,c5,c2_literal" if world == 1 else "c5"
    for name in [w for w in want.split(",") if w and w != "none"]:
        c = dict(BASELINE_CONFIGS[name])
        if name == "c4":
            c["envs"] = args.c4_envs
        try:
            r, e_ = run_config(c, K, Wm, rank, world, local_rank, "hwc_uint8", None, gather=(name == "c5"), gather_impl=args.gather)
            e_.close()
            del e_
            extra[name] = r
        except Exception as ex:
            extra[name] = {"error": f"{type(ex).__name__}: {ex}"}
        torch.cuda.empty_cache()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    traffic = None
    tp = os.path.join(ROOT, "profiles", "render_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        if tj.get("envs") == E and tj.get("width") == W and tj.get("map") == args.map:
            traffic = tj.get("dram_bytes_per_launch")
    res["roofline"]["traffic"] = traffic
    line = {
        "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64 logic / f32 raster / u8 obs", "data": "synthetic", "config": config,
        "clocks": sampler.summary(), "e2e": e2e, "gpu_launches": res["gpu_launches"], "roofline": res["roofline"],
        "kernel_ms": res["kernel_ms"], "parity_unpinned": PARITY_UNPINNED, "numa": numa,
        "baseline_is": "cpu_baseline / --impl reference = C port of the reference's CPU path (oracle/), not the Pyglet reference (cannot run here)",
    }
    if e2e_resized is not None:
        line["e2e_resized"] = e2e_resized
    if extra:
        line["configs"] = extra
    if not args.no_cpu_baseline:
        val, secs, used, desc = cpu_reference_run(args.map.split(",")[0], W, H, 4, 1, args.cpu_sample_envs, cores)
        line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": used, "kind": "port", "sample": desc}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
