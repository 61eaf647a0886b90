#!/usr/bin/env python3
"""Generate tests/golden/*.npz by executing the REFERENCE's own code (via oracle/refstub.py).

Run in the build container only (needs /root/reference):   python oracle/make_golden.py
The fixtures it writes are committed; the GPU box has no /root/reference and only reads them.

Files written
  logic_<map>.npz      poses -> tile coords, drivable, valid_pose (sf 1.0 / 1.3), collision, proximity,
                       lane pose, reward / done / done_code          (reference: simulator.py, collision.py, graphics.py)
  action_map.npz       DuckietownEnv.step [vel, steer] -> wheel duty  (envs/duckietown_env.py:36-59)
  reset_<map>.npz      Simulator.reset() outputs per seed, domain_rand off/on (simulator.py:528-763)
  fisheye.npz          Distortion LUT digest, sub-sampled LUT, one remapped test image (distortion.py)
  gltrace_<map>.npz    what the reference's own _render_img / _init_vlists / WorldObj.render / reset() lighting ask
                       OpenGL to do, recorded call by call (oracle/gltrace.py): per frame the projection arguments,
                       look-at, model-view of every draw, GL_LIGHT0 (eye-space position, ambient, diffuse), current
                       colour, bound texture, draw order; the vertex lists            (simulator.py:386-527, 564-586,
                       1707-1951; objects.py:123-148)
  wrapper_interface.npz  observation spaces / shapes of the reference's PyTorchObsWrapper + ResizeWrapper around an
                       object with the product Simulator's spaces                      (wrappers.py:93-141)
  objmesh.npz          ObjMesh's extents and per-corner attributes for the synthetic OBJ of tests/test_obj_loader.py
                       (objmesh.py:65-293)
"""
from __future__ import annotations

import hashlib
import functools
import os
from unittest import mock
import sys

import numpy as np
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import refstub  # noqa: E402
from gym_duckietown_b200 import assets, maps  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
MAPS = ["small_loop", "loop_obstacles", "udem1"]


def raw_map(name):
    with open(os.path.join(ROOT, "gym-duckietown_b200", "maps", f"{name}.yaml")) as f:
        return yaml.safe_load(f)


def extents_for(raw):
    objs = raw.get("objects") or []
    descs = objs.values() if isinstance(objs, dict) else objs
    ext = {}
    for o in descs:
        k = o["kind"]
        m = assets.get_mesh(k)
        ext["sign_generic" if k.startswith("sign") else k] = (m.min_coords, m.max_coords)
    return ext


def sample_poses(md: maps.MapData, n: int, rng) -> np.ndarray:
    """Mixture: anywhere (incl. off-grid), on drivable tiles, hugging obstacles, exact tile edges."""
    ts, W, H = md.tile_size, md.grid_w, md.grid_h
    out = []
    for k in range(n):
        mode = k % 8
        if mode == 0:
            x, z = rng.uniform(-0.5, W + 0.5) * ts, rng.uniform(-0.5, H + 0.5) * ts
        elif mode in (1, 2, 3, 4):
            i, j = md.drivable_tiles[rng.integers(0, len(md.drivable_tiles))]
            x, z = rng.uniform(i, i + 1) * ts, rng.uniform(j, j + 1) * ts
        elif mode in (5, 6) and md.n_coll:
            c = md.coll_centers[rng.integers(0, md.n_coll)]
            r = rng.uniform(0, 0.35)
            a = rng.uniform(0, 2 * np.pi)
            x, z = c[0] + r * np.cos(a), c[2] + r * np.sin(a)
        elif mode == 7:
            i, j = md.drivable_tiles[rng.integers(0, len(md.drivable_tiles))]
            x, z = i * ts, rng.uniform(j, j + 1) * ts  # exactly on a tile boundary in x
            if k % 16 == 15:
                x, z = rng.uniform(i, i + 1) * ts, (j + 1) * ts
        else:
            i, j = md.drivable_tiles[rng.integers(0, len(md.drivable_tiles))]
            x, z = rng.uniform(i, i + 1) * ts, rng.uniform(j, j + 1) * ts
        ang = rng.uniform(-np.pi, np.pi) if k % 5 else rng.choice([0.0, np.pi / 2, np.pi, -np.pi / 2, 2 * np.pi])
        out.append((x, z, ang))
    return np.array(out)


def gen_logic(name: str, n=1536, seed=7):
    raw = raw_map(name)
    md = maps.load_map(name)
    sim = refstub.build_reference_sim(raw, extents_for(raw))
    S, C, G, O = refstub.modules()
    from gym_duckietown.exceptions import NotInLane

    rng = np.random.default_rng(seed)
    poses = sample_poses(md, n, rng)
    steps = rng.integers(0, 4, n)  # 0 -> step_count = max_steps (max-steps branch), else small
    rec = {k: [] for k in ("ti", "tj", "drv", "valid10", "valid13", "coll1", "coll2", "prox", "inlane", "dist",
                           "dot", "ang", "reward", "done", "code", "corners")}
    for (x, z, a), st in zip(poses, steps):
        pos = np.array([x, 0.0, z])
        i, j = sim.get_grid_coords(pos)
        rec["ti"].append(i); rec["tj"].append(j)
        rec["drv"].append(sim._drivable_pos(pos))
        rec["valid10"].append(sim._valid_pose(pos, a))
        rec["valid13"].append(sim._valid_pose(pos, a, safety_factor=1.3))
        corners = S.get_agent_corners(pos, a)
        rec["corners"].append(corners)
        rec["coll1"].append(sim._collision(corners))  # run_tests.py:50 usage (offset once)
        rec["coll2"].append(sim._collision(S.get_agent_corners(S._actual_center(pos, a), a)))  # S:1502,1521
        rec["prox"].append(sim.proximity_penalty2(pos, a))
        try:
            lp = sim.get_lane_pos2(pos, a)
            rec["inlane"].append(True); rec["dist"].append(lp.dist); rec["dot"].append(lp.dot_dir)
            rec["ang"].append(lp.angle_rad)
        except NotInLane:
            rec["inlane"].append(False); rec["dist"].append(np.nan); rec["dot"].append(np.nan)
            rec["ang"].append(np.nan)
        sim.cur_pos, sim.cur_angle = pos, a
        sim.step_count = sim.max_steps if st == 0 else int(st)
        d = sim._compute_done_reward()
        rec["reward"].append(float(d.reward)); rec["done"].append(d.done)
        rec["code"].append({"in-progress": 0, "invalid-pose": 1, "max-steps-reached": 2}[d.done_code])
    arrs = {k: np.array(v) for k, v in rec.items()}
    arrs["poses"] = poses
    arrs["step_count"] = np.where(steps == 0, sim.max_steps, steps).astype(np.int32)
    arrs["max_steps"] = np.int32(sim.max_steps)
    # load-time arrays, to pin maps.py against the reference's own map interpretation
    arrs["ref_curves"] = np.concatenate([t["curves"] for t in sim.drivable_tiles], 0)
    arrs["ref_drivable_ij"] = np.array([t["coords"] for t in sim.drivable_tiles])
    if md.n_coll:
        arrs["ref_coll_corners"] = np.asarray(sim.collidable_corners)
        arrs["ref_coll_norms"] = np.asarray(sim.collidable_norms)
        arrs["ref_coll_centers"] = np.asarray(sim.collidable_centers)
        arrs["ref_coll_radii"] = np.asarray(sim.collidable_safety_radii)
    np.savez_compressed(os.path.join(OUT, f"logic_{name}.npz"), **arrs)
    print(f"logic_{name}: {n} poses, done={arrs['done'].mean():.2f} inlane={arrs['inlane'].mean():.2f} "
          f"coll={arrs['coll2'].mean():.3f}")


def gen_action_map(n=512, seed=11):
    refstub.install()
    from gym_duckietown.envs import duckietown_env as E
    import gym_duckietown.simulator as S

    rng = np.random.default_rng(seed)
    acts = rng.uniform(-1, 1, (n, 2)).astype(np.float32)
    wd = rng.uniform(0.0918, 0.1122, n)
    cfgs = [(1.0, 0.0, 0.0318, 27.0, 1.0), (0.8, 0.05, 0.03, 25.0, 0.9)]
    got = np.zeros((len(cfgs), n, 2))
    captured = {}

    def fake_step(self, vels):
        captured["v"] = np.array(vels, dtype=np.float64)
        return None, 0.0, False, {}

    orig = S.Simulator.step
    S.Simulator.step = fake_step
    try:
        for c, (gain, trim, radius, k, limit) in enumerate(cfgs):
            env = object.__new__(E.DuckietownEnv)
            env.gain, env.trim, env.radius, env.k, env.limit = gain, trim, radius, k, limit
            for q in range(n):
                env.wheel_dist = np.array(wd[q])
                env.step(acts[q])
                got[c, q] = captured["v"]
    finally:
        S.Simulator.step = orig
    np.savez_compressed(os.path.join(OUT, "action_map.npz"), actions=acts, wheel_dist=wd, cfgs=np.array(cfgs),
                        vels=got)
    print("action_map:", got.shape)


RESET_KEYS = ["cur_pos", "cur_angle", "wheel_dist", "cam_height", "cam_angle", "cam_fov_y", "camera_noise",
              "horizon_color", "ground_color", "light_pos", "trim", "obj_visible"]


def gen_reset(name: str, seeds=range(24)):
    raw = raw_map(name)
    S, C, G, O = refstub.modules()
    out = {}
    for dr in (False, True):
        rows = {k: [] for k in RESET_KEYS + ["ambient", "diffuse"]}
        for seed in seeds:
            sim = refstub.build_reference_sim(raw, extents_for(raw), domain_rand=dr, seed=int(seed))
            captured = []
            S.gl.glLightfv = lambda light, pname, arr: captured.append(arr)
            # ctypes arrays are mocked: (gl.GLfloat * 4)(*vals) -> capture through a fake GLfloat
            class _GLf:
                def __mul__(self, n):
                    return lambda *v: np.array(v, dtype=np.float32)
            S.gl.GLfloat = _GLf()
            for episode in range(2):  # two consecutive episodes from one stream
                captured.clear()
                sim.reset()
                rows["cur_pos"].append(np.array(sim.cur_pos, float)); rows["cur_angle"].append(float(sim.cur_angle))
                rows["wheel_dist"].append(float(sim.wheel_dist)); rows["cam_height"].append(float(sim.cam_height))
                rows["cam_angle"].append(float(sim.cam_angle[0])); rows["cam_fov_y"].append(float(sim.cam_fov_y))
                rows["camera_noise"].append(np.array(sim.randomization_settings["camera_noise"], float))
                rows["horizon_color"].append(np.array(sim.horizon_color, float))
                rows["ground_color"].append(np.array(sim.ground_color, float))
                lp = np.zeros(4); lp[:len(captured[0])] = captured[0]
                rows["light_pos"].append(lp)
                rows["ambient"].append(np.array(captured[1], float)); rows["diffuse"].append(np.array(captured[2], float))
                rows["trim"].append(float(sim.randomization_settings["trim"][0]))
                rows["obj_visible"].append(np.array([o.visible for o in sim.objects], bool))
        for k, v in rows.items():
            out[f"{'dr' if dr else 'nodr'}_{k}"] = np.array(v)
    out["seeds"] = np.array(list(seeds))
    np.savez_compressed(os.path.join(OUT, f"reset_{name}.npz"), **out)
    print(f"reset_{name}: seeds={len(out['seeds'])} x 2 episodes x (dr off/on)")


CUSTOM_DR = {   # a user's randomization_config_fp: other ranges, a shuffled-in unknown key before and after the known ones
    "aa_first": {"type": "int", "low": 0, "high": 10, "size": 2},
    "horz_mode": {"type": "int", "low": 1, "high": 3},
    "light_pos": {"type": "uniform", "low": [-100, 150, -100], "high": [100, 250, 100], "size": 3},
    "camera_noise": {"type": "uniform", "low": -0.01, "high": 0.01, "size": 3},
    "trim": {"type": "normal", "loc": 0.01, "scale": 0.05},
    "camera_height": {"type": "uniform", "low": 0.8, "high": 1.0},
    "camera_angle": {"type": "uniform", "low": 0.9, "high": 1.1},
    "camera_fov_y": {"type": "uniform", "low": 0.95, "high": 1.05},
    "zz_extra": {"type": "uniform", "low": 0.0, "high": 1.0, "size": 5},
}
CUSTOM_SIM = dict(num_tris_distractors=5, color_sky=[0.2, 0.5, 0.7], color_ground=[0.3, 0.25, 0.2])


def gen_reset_custom(name="loop_obstacles", seeds=range(40, 56)):
    """reset() with Randomizer(randomization_config_fp=<custom table>) (randomizer.py:19-33) and non-default
    num_tris_distractors / color_sky / color_ground (S:226-230), domain_rand and dynamics_rand on."""
    raw = raw_map(name)
    S, C, G, O = refstub.modules()
    rows = {k: [] for k in RESET_KEYS + ["ambient", "diffuse"]}
    for seed in seeds:
        sim = refstub.build_reference_sim(raw, extents_for(raw), domain_rand=True, seed=int(seed), dynamics_rand=True)
        sim.randomizer.randomization_config = dict(CUSTOM_DR)
        sim.randomizer.keys = sorted(set(list(CUSTOM_DR.keys()) + list(sim.randomizer.default_config.keys())))
        sim.num_tris_distractors = CUSTOM_SIM["num_tris_distractors"]
        sim.color_sky, sim.color_ground = list(CUSTOM_SIM["color_sky"]), list(CUSTOM_SIM["color_ground"])
        captured = []
        S.gl.glLightfv = lambda light, pname, arr: captured.append(arr)

        class _GLf:
            def __mul__(self, n):
                return lambda *v: np.array(v, dtype=np.float32)
        S.gl.GLfloat = _GLf()
        for episode in range(2):
            captured.clear()
            sim.reset()
            rows["cur_pos"].append(np.array(sim.cur_pos, float)); rows["cur_angle"].append(float(sim.cur_angle))
            rows["wheel_dist"].append(float(sim.wheel_dist)); rows["cam_height"].append(float(np.ravel(sim.cam_height)[0]))
            rows["cam_angle"].append(float(np.ravel(sim.cam_angle[0])[0])); rows["cam_fov_y"].append(float(np.ravel(sim.cam_fov_y)[0]))
            rows["camera_noise"].append(np.array(sim.randomization_settings["camera_noise"], float))
            rows["horizon_color"].append(np.array(sim.horizon_color, float))
            rows["ground_color"].append(np.array(sim.ground_color, float))
            lp = np.zeros(4); lp[:len(captured[0])] = captured[0]
            rows["light_pos"].append(lp)
            rows["ambient"].append(np.array(captured[1], float)); rows["diffuse"].append(np.array(captured[2], float))
            rows["trim"].append(float(sim.randomization_settings["trim"][0]))
            rows["obj_visible"].append(np.array([o.visible for o in sim.objects], bool))
    out = {f"dr_{k}": np.array(v) for k, v in rows.items()}
    out["seeds"] = np.array(list(seeds))
    import json
    out["config_json"] = json.dumps(CUSTOM_DR)
    out["sim_json"] = json.dumps(CUSTOM_SIM)
    np.savez_compressed(os.path.join(OUT, f"reset_customdr_{name}.npz"), **out)
    print(f"reset_customdr_{name}: {len(out['seeds'])} seeds x 2 episodes")


def gen_reset_start(name="udem1", seeds=range(12)):
    """reset() with a fixed start: `user_tile_start` (S:659-666, beats the map's start_tile, no tile draw), the map's
    `start_tile` (S:668-669) and `start_pose` (S:679-686, no spawn loop at all) — as executed by the reference."""
    import copy
    raw = raw_map(name)
    out = {"seeds": np.array(list(seeds))}
    cases = {"user": (raw, dict(user_tile_start=(1, 1))),
             "tile": (dict(copy.deepcopy(raw), start_tile=[3, 1]), {}),
             "pose": (dict(copy.deepcopy(raw), start_tile=[3, 1], start_pose=[[0.21, 0.0, 0.33], 1.4]), {})}
    for tag, (mp, kw) in cases.items():
        pos, ang = [], []
        for seed in seeds:
            sim = refstub.build_reference_sim(mp, extents_for(mp), domain_rand=False, seed=int(seed), **kw)
            for episode in range(2):
                sim.reset()
                pos.append(np.array(sim.cur_pos, float)); ang.append(float(sim.cur_angle))
        out[f"{tag}_cur_pos"], out[f"{tag}_cur_angle"] = np.array(pos), np.array(ang)
    out["start_tile"], out["start_pose"], out["user_tile_start"] = np.array([3, 1]), np.array([0.21, 0.0, 0.33, 1.4]), np.array([1, 1])
    np.savez_compressed(os.path.join(OUT, f"reset_start_{name}.npz"), **out)
    print(f"reset_start_{name}: {len(out['seeds'])} seeds x 2 episodes x (user_tile_start, start_tile, start_pose)")


def gen_helpers(n=256, seed=9):
    """Module-level helpers of simulator.py that user scripts import (S:2056-2118)."""
    S, C, G, O = refstub.modules()
    rng = np.random.default_rng(seed)
    poses = np.stack([rng.uniform(0, 5, n), np.zeros(n), rng.uniform(0, 5, n)], 1)
    angles = rng.uniform(-2 * np.pi, 2 * np.pi, n)
    np.savez_compressed(os.path.join(OUT, "helpers.npz"), poses=poses, angles=angles,
                        dir_vec=np.array([S.get_dir_vec(a) for a in angles]),
                        right_vec=np.array([S.get_right_vec(a) for a in angles]),
                        center=np.array([S._actual_center(p, a) for p, a in zip(poses, angles)]),
                        corners=np.array([S.get_agent_corners(p, a) for p, a in zip(poses, angles)]))
    print(f"helpers: {n} poses")


def gen_fisheye():
    refstub.install()
    from gym_duckietown.distortion import Distortion

    d = Distortion()
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (480, 640, 3), dtype=np.uint8)
    out = d.distort(img)
    rx, ry = d.rmapx.astype(np.float32), d.rmapy.astype(np.float32)
    np.savez_compressed(
        os.path.join(OUT, "fisheye.npz"),
        sha_rmapx=hashlib.sha256(rx.tobytes()).hexdigest(), sha_rmapy=hashlib.sha256(ry.tobytes()).hexdigest(),
        rmapx_sub=rx[::8, ::8], rmapy_sub=ry[::8, ::8], img_seed=5,
        out_sha=hashlib.sha256(out.tobytes()).hexdigest(), out_sub=out[::8, ::8],
        new_camera_matrix=d.new_camera_matrix)
    print("fisheye: holes-free LUT", np.isnan(rx).sum() == 0, "out mean", out.mean())


def gen_dynamic(name: str, steps=900, seed=21):
    """Dynamic obstacles (SURVEY 8f-2): DuckieObj / DuckiebotObj stepped by the reference's own code
    (objects.py:180-432, update loop simulator.py:1570-1584), plus agent collision / proximity queries against
    them.  domain_rand=False, so the only global-RNG draw is DuckieObj.wiggle (recorded as an input)."""
    raw = raw_map(name)
    md = maps.load_map(name)
    np.random.seed(seed)   # objects.py draws from the GLOBAL numpy RNG (SURVEY app. B-10)
    sim = refstub.build_reference_sim(raw, extents_for(raw))
    S, C, G, O = refstub.modules()
    dyn = [o for o in sim.objects if not o.static]
    rec = {k: [] for k in ("pos", "angle", "y_rot", "corners", "active")}
    rng = np.random.default_rng(seed)
    q_pose, q_coll, q_prox, q_step = [], [], [], []
    wiggle = np.array([float(np.ravel(getattr(o, "wiggle", 0.0))[0]) for o in dyn])
    for t in range(steps):
        for obj in sim.objects:   # S:1570-1584
            if obj.kind == "duckiebot":
                if not obj.static:
                    obj.step_duckiebot(sim.delta_time, sim.closest_curve_point, [])
            else:
                obj.step(sim.delta_time)
        rec["pos"].append([np.array(o.pos, float) for o in dyn])
        rec["angle"].append([float(o.angle) for o in dyn])
        rec["y_rot"].append([float(o.y_rot) for o in dyn])
        rec["corners"].append([np.array(o.obj_corners, float) for o in dyn])
        rec["active"].append([bool(getattr(o, "pedestrian_active", False)) for o in dyn])
        if t % 5 == 0:   # probe agent poses around a dynamic object
            o = dyn[rng.integers(len(dyn))]
            r, a = rng.uniform(0, 0.3), rng.uniform(0, 2 * np.pi)
            pos = np.array([o.pos[0] + r * np.cos(a), 0.0, o.pos[2] + r * np.sin(a)])
            ang = rng.uniform(-np.pi, np.pi)
            q_pose.append((pos[0], pos[2], ang)); q_step.append(t)
            q_coll.append(sim._collision(S.get_agent_corners(pos, ang)))
            q_prox.append(sim.proximity_penalty2(pos, ang))
    out = {k: np.array(v) for k, v in rec.items()}
    out.update(wiggle=wiggle, q_pose=np.array(q_pose), q_step=np.array(q_step), q_coll=np.array(q_coll), q_prox=np.array(q_prox),
               dyn_index=np.array([sim.objects.index(o) for o in dyn]))
    np.savez_compressed(os.path.join(OUT, f"dynamic_{name}.npz"), **out)
    print(f"dynamic_{name}: {len(dyn)} dynamic objects x {steps} steps, collisions {np.mean(q_coll):.2f}, "
          f"active {out['active'].mean():.2f}")


def gen_trafficlight(name="loop_trafficlights", steps=1300, seed=5):
    """TrafficLightObj (objects.py:434-476) stepped by the reference's own code: pattern per light, and which card
    the SHARED mesh shows (every light assigns mesh.textures[0]; the last writer wins).  Two runs: the
    non-randomized defaults (freq 5, pattern 0) and domain_rand=True, where the reference draws freq / pattern from
    the global numpy RNG at construction (recorded as inputs)."""
    raw = raw_map(name)
    out = {}
    for tag, dr in (("plain", False), ("dr", True)):
        np.random.seed(seed)
        S, C, G, O = refstub.modules()
        # graphics.load_texture is lru_cached per path (G:69); under the pyglet mock every call returns the same
        # MagicMock, so give each path its own token
        with mock.patch.object(O, "load_texture", functools.lru_cache(maxsize=None)(lambda path, *a, **k: ("tex", path))), \
                mock.patch.object(O, "get_resource_path", lambda fn: fn):     # duckietown_world is a mock too
            sim = refstub.build_reference_sim(raw, extents_for(raw), domain_rand=dr)
        tls = [o for o in sim.objects if isinstance(o, O.TrafficLightObj)]
        assert len({id(o.mesh) for o in tls}) == 1 and tls[0].texs[0] is not tls[0].texs[1]

        def shown():
            tex = tls[0].mesh.textures[0]
            return [j for o in tls for j in (0, 1) if o.texs[j] is tex][0]
        out[f"{tag}_freq"] = np.array([o.freq for o in tls])
        out[f"{tag}_pattern0"] = np.array([o.pattern for o in tls])
        out[f"{tag}_shown0"] = np.array(shown())
        pat, shw = [], []
        for t in range(steps):
            for obj in sim.objects:   # S:1570-1584
                obj.step(sim.delta_time)
            pat.append([o.pattern for o in tls])
            shw.append(shown())
        out[f"{tag}_pattern"], out[f"{tag}_shown"] = np.array(pat, np.int8), np.array(shw, np.int8)
        out["tl_index"] = np.array([sim.objects.index(o) for o in tls])
        print(f"trafficlight_{name}[{tag}]: freq {out[f'{tag}_freq']}, pattern0 {out[f'{tag}_pattern0']}, "
              f"flips {np.abs(np.diff(out[f'{tag}_pattern'], axis=0)).sum(0)}, shown flips {np.abs(np.diff(shw)).sum()}")
    np.savez_compressed(os.path.join(OUT, f"trafficlight_{name}.npz"), **out)


def gen_wrappers(seed=21):
    """The reference's own wrapper classes (src/gym_duckietown/wrappers.py, learning/utils/wrappers.py) executed on
    canned frames / rewards / actions -> tests/golden/wrappers.npz.  A stand-in env hands them the frames: what is
    recorded is exactly what their observation() / reward() / action() / step() code returns."""
    refstub.install()
    sys.path.insert(0, "/root/reference")
    import importlib
    W = importlib.import_module("gym_duckietown.wrappers")
    LW = importlib.import_module("learning.utils.wrappers")
    spaces = sys.modules["gym.spaces"]
    rng = np.random.default_rng(seed)
    out = {}
    for tag, (h, w_) in {"160x120": (120, 160), "640x480": (480, 640)}.items():
        frames = rng.integers(0, 256, (3, h, w_, 3), dtype=np.uint8)
        # smooth content too (renders are smooth; noise is the hard case for a fixed-point filter)
        yy, xx = np.mgrid[0:h, 0:w_]
        frames[2] = np.stack([(xx * 255 // w_), (yy * 255 // h), ((xx + yy) * 255 // (h + w_))], -1).astype(np.uint8)

        class Env:   # what DuckietownEnv looks like to a wrapper
            metadata, reward_range = {}, (-1000, 1000)
            action_space = spaces.Box(low=-1, high=1, shape=(2,), dtype=np.float32)
            observation_space = spaces.Box(low=np.zeros((h, w_, 3), np.uint8), high=np.full((h, w_, 3), 255, np.uint8),
                                           shape=(h, w_, 3), dtype=np.uint8)
            k = 0
            actions = []

            @property
            def unwrapped(self):
                return self

            def reset(self):
                return frames[0]

            def step(self, a):
                Env.actions.append(np.array(a, dtype=float))
                Env.k += 1
                return frames[Env.k % 3], -1000.0 if Env.k % 3 == 0 else float(Env.k) - 2.5, False, {}

        # the test regenerates the frames from the seed (default_rng(seed), same draw order) and checks this digest
        out[f"frames_sha_{tag}"] = hashlib.sha256(frames.tobytes()).hexdigest()
        digest = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
        pt = W.PyTorchObsWrapper(Env())
        out[f"pytorch_sha_{tag}"] = digest(np.stack([pt.observation(f) for f in frames]))
        assert tuple(pt.observation_space.shape) == (3, w_, h)
        for rw, rh in ((80, 80), (84, 84), (64, 48)):
            rz = W.ResizeWrapper(W.PyTorchObsWrapper(Env()), resize_w=rw, resize_h=rh)
            got = [rz.reset()] + [rz.step([0.0, 0.0])[0] for _ in range(2)]
            Env.k = 0
            out[f"resize_{tag}_{rw}x{rh}"] = np.stack(got)        # [3][C][rw][rh] as the wrapper returns them
        img = LW.ImgWrapper(Env())
        out[f"img_sha_{tag}"] = digest(np.stack([img.observation(f) for f in frames]))
        nm = LW.NormalizeWrapper(Env())
        nf = np.stack([nm.observation(f) for f in frames[:1]])
        out[f"norm_dtype_{tag}"] = str(nf.dtype)
        out[f"norm_f32_sha_{tag}"] = digest(nf.astype(np.float32))
    rewards = np.array([-1000.0, -999.0, -3.2, 0.0, 1e-9, 0.7, 12.5])
    dt = LW.DtRewardWrapper(Env())
    out["rewards"], out["dt_rewards"] = rewards, np.array([dt.reward(r) for r in rewards])
    aw = LW.ActionWrapper(Env())
    acts = rng.uniform(-1, 1, (16, 2))
    out["actions"], out["scaled_actions"] = acts, np.array([aw.action(a) for a in acts])
    dw = W.DiscreteWrapper(Env())
    out["discrete_actions"] = np.array([dw.action(k) for k in range(3)])
    out["seed"] = np.int64(seed)
    np.savez_compressed(os.path.join(OUT, "wrappers.npz"), **out)
    print("wrappers:", sorted(out))


def gen_wrapper_interface():
    """The reference's PyTorchObsWrapper and ResizeWrapper (wrappers.py:93-141), unmodified, wrapped around an object
    that carries the product Simulator's spaces and step / reset signature -> tests/golden/wrapper_interface.npz: the
    observation spaces they declare and the shapes they return."""
    refstub.install()
    import importlib
    W = importlib.import_module("gym_duckietown.wrappers")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_reference_wrappers import StandIn

    pt = W.PyTorchObsWrapper(StandIn())
    first = pt.reset()
    second = pt.step([0, 0])[0]
    rz = W.ResizeWrapper(pt, resize_w=84, resize_h=84)
    out = {"obs_shapes": np.array([first.shape, second.shape])}
    for tag, sp in (("pytorch", pt.observation_space), ("resize", rz.observation_space)):
        out[f"{tag}_shape"] = np.array(sp.shape)
        out[f"{tag}_low"], out[f"{tag}_high"] = np.array(sp.low).ravel()[:1], np.array(sp.high).ravel()[:1]
        out[f"{tag}_dtype"] = np.dtype(sp.dtype).str
    out["resize_reset_shape"] = np.array(rz.reset().shape)
    np.savez_compressed(os.path.join(OUT, "wrapper_interface.npz"), **out)
    print("wrapper_interface:", {k: np.asarray(v).tolist() for k, v in out.items()})


def gen_objmesh():
    """The reference's ObjMesh loader (objmesh.py:65-293) on the synthetic OBJ / MTL pair of tests/test_obj_loader.py
    -> tests/golden/objmesh.npz: extents and the per-corner attributes it hands pyglet."""
    import tempfile
    refstub.install()
    import gym_duckietown.objmesh as M
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_obj_loader import MTL, OBJ, source_digest

    captured = []

    def vertex_list(n, *attrs):
        captured.append({name: np.array(data, dtype=np.float32) for name, data in attrs})
        return object()

    with tempfile.TemporaryDirectory() as d:
        for name, text in (("prop.obj", OBJ), ("prop.mtl", MTL)):
            with open(os.path.join(d, name), "w") as f:
                f.write(text)

        def resource(name):
            p = os.path.join(d, name)
            if not os.path.exists(p):
                raise KeyError(name)
            return p

        M.pyglet.graphics.vertex_list = vertex_list
        M.get_resource_path = resource
        ref = M.ObjMesh(os.path.join(d, "prop.obj"), "prop")
    np.savez_compressed(
        os.path.join(OUT, "objmesh.npz"), source_sha=source_digest(), min_coords=ref.min_coords, max_coords=ref.max_coords,
        tri_pos=np.concatenate([c["v3f"].reshape(-1, 3, 3) for c in captured]),
        tri_nrm=np.concatenate([c["n3f"].reshape(-1, 3, 3) for c in captured]),
        tri_uv=np.concatenate([c["t2f"].reshape(-1, 3, 2) for c in captured]),
        tri_col=np.concatenate([c["c3f"].reshape(-1, 3, 3) for c in captured]))
    print(f"objmesh: {sum(len(c['v3f']) // 9 for c in captured)} triangles in {len(captured)} vertex lists")


def gen_gltrace(name: str, seeds=(11, 12, 13), poses_per_episode=8, width=160, height=120):
    """Run the reference's render path against the recording GL (oracle/gltrace.py): reset() + a short walk, twice per
    seed (the second episode captures GL_LIGHT0 under the previous frame's model-view, S:581), domain_rand off and on."""
    import gltrace
    rec = gltrace.GLRecorder()
    gltrace.attach(rec)
    raw = raw_map(name)
    S, C, G, O = refstub.modules()
    frames, draws = [], []
    vl = {}
    tex_names = []

    def tex_index(tid):
        if tid is None:
            return -1
        nm = rec.tex_names[tid][0]
        if nm not in tex_names:
            tex_names.append(nm)
        return tex_names.index(nm)

    mesh_kinds = []
    distractors = []
    for dr in (False, True):
        for seed in seeds:
            sim = gltrace.make_sim(rec, raw, extents_for(raw), domain_rand=dr, seed=int(seed), width=width, height=height)
            if not vl:
                vl = dict(road_v=sim.road_vlist.attrs["v"], road_t=sim.road_vlist.attrs["t"], road_n=sim.road_vlist.attrs["n"],
                          road_c=sim.road_vlist.attrs["c"], ground_v=sim.ground_vlist.attrs["v"])
            rng = np.random.default_rng(1000 + seed)
            for episode in range(2):
                rec.take()
                sim.reset()
                distractors.append(np.concatenate([sim.tri_vlist.attrs["v"], sim.tri_vlist.attrs["c"]], 1))
                modes = [0] * (poses_per_episode + 1)
                if episode == 1:
                    modes += [2] + ([1] if not dr else [])   # one top_down frame; one segment frame (DR off: the DR texture
                                                             # pick in get_texture calls rng.randint, absent from a Generator)
                for k, mode in enumerate(modes):
                    if k > 0 and mode == 0:   # a short walk from the spawn pose: rendering does not need a valid pose
                        d = S.get_dir_vec(sim.cur_angle)
                        sim.cur_pos = np.array(sim.cur_pos, float) + d * rng.uniform(0.02, 0.2)
                        sim.cur_angle = float(sim.cur_angle) + rng.uniform(-0.5, 0.5)
                        rec.take()
                        sim.render_obs()
                    elif mode == 1:
                        rec.take()
                        sim.render_obs(segment=True)
                    elif mode == 2:
                        rec.take()
                        sim._render_img(width, height, sim.multi_fbo, sim.final_fbo, sim.img_array, top_down=True, segment=False)
                    ev = rec.take()
                    lights = [e for e in ev if e["kind"] == "light"]
                    clear = [e for e in ev if e["kind"] == "clear"][-1]
                    look = [e for e in ev if e["kind"] == "lookat"][-1]
                    dl = [e for e in ev if e["kind"] == "draw"]
                    f = dict(dr=dr, seed=seed, episode=episode, k=k, mode=mode, pos=np.array(sim.cur_pos, float), angle=float(sim.cur_angle),
                             clear=clear["color"], persp=np.array(rec.perspective), eye=look["eye"], center=look["center"],
                             view=look["modelview"].reshape(-1), proj=dl[0]["projection"].reshape(-1),
                             light_eye=dl[0]["light_pos_eye"], light_ambient=dl[0]["light_ambient"],
                             light_diffuse=dl[0]["light_diffuse"], light_model_ambient=dl[0]["light_model_ambient"],
                             light_raw=(lights[0]["values"] if lights else np.full(4, np.nan)),
                             flags=np.array([dl[0]["lighting"], dl[0]["light0"], dl[0]["color_material"], dl[0]["normalize"],
                                             dl[0]["rescale_normal"]], np.int8),
                             cam_height=float(np.asarray(sim.cam_height).reshape(-1)[0]),
                             cam_angle=float(np.asarray(sim.cam_angle[0]).reshape(-1)[0]),
                             cam_fov_y=float(np.asarray(sim.cam_fov_y).reshape(-1)[0]),
                             camera_noise=np.array(sim.randomization_settings["camera_noise"], float),
                             horizon=np.array(sim.horizon_color, float), ground=np.array(sim.ground_color, float),
                             draw0=len(draws), visible=np.array([o.visible for o in sim.objects], bool))
                    for e in dl:
                        if e["what"] == "vlist":
                            v = rec.vlists[e["id"]]
                            kind = 0 if v is sim.ground_vlist else (1 if v is sim.tri_vlist else 2)
                            sub = -1
                        else:
                            kind = 3
                            if e["id"] not in mesh_kinds:
                                mesh_kinds.append(e["id"])
                            sub = mesh_kinds.index(e["id"])
                        tid = e["texture"]
                        draws.append(dict(frame=len(frames), kind=kind, sub=sub, mv=e["modelview"].reshape(-1), color=e["color"],
                                          tex=tex_index(tid), lit=e["lighting"],
                                          tex_seg=bool(tid is not None and rec.tex_names[tid][1]), mesh_seg=bool(e.get("segment", False))))
                    f["ndraws"] = len(draws) - f["draw0"]
                    frames.append(f)
    out = {f"f_{k}": np.array([fr[k] for fr in frames]) for k in frames[0] if k != "visible"}
    nobj = max(len(fr["visible"]) for fr in frames)
    out["f_visible"] = np.array([np.pad(fr["visible"], (0, nobj - len(fr["visible"]))) for fr in frames])
    out.update({f"d_{k}": np.array([d[k] for d in draws]) for k in draws[0]})
    out.update(vl)
    out["distractors"] = np.array(distractors)
    out["tex_names"] = np.array(tex_names)
    out["mesh_kinds"] = np.array(mesh_kinds if mesh_kinds else [""])
    out["width"], out["height"] = np.int32(width), np.int32(height)
    np.savez_compressed(os.path.join(OUT, f"gltrace_{name}.npz"), **out)
    print(f"gltrace_{name}: {len(frames)} frames, {len(draws)} draws, textures {tex_names}, meshes {mesh_kinds}")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "customdr":
        os.makedirs(OUT, exist_ok=True)
        gen_reset_custom()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "wrappers":
        os.makedirs(OUT, exist_ok=True)
        gen_wrappers()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "interfaces":
        os.makedirs(OUT, exist_ok=True)
        gen_wrapper_interface()
        gen_objmesh()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "gltrace":
        os.makedirs(OUT, exist_ok=True)
        for m in MAPS:
            gen_gltrace(m)
        sys.exit(0)
    os.makedirs(OUT, exist_ok=True)
    for m in MAPS:
        gen_logic(m)
    gen_action_map()
    for m in ("small_loop", "loop_obstacles", "udem1"):
        gen_reset(m)
    gen_fisheye()
    for m in ("loop_pedestrians", "loop_dyn_duckiebots"):
        gen_dynamic(m)
    gen_trafficlight()
    gen_reset_start()
    gen_reset_custom()
    gen_helpers()
    gen_wrappers()
    gen_wrapper_interface()
    gen_objmesh()
    for m in MAPS:
        gen_gltrace(m)
