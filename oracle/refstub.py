"""Stub-import harness: run the reference's OWN numpy arithmetic without its missing dependencies.

TEST INFRASTRUCTURE ONLY.  Nothing in the product package imports this file.  It is used by
``oracle/make_golden.py``, where the reference source tree is present, to produce the fixtures
under ``tests/golden/``; the tests only read those fixtures.

What it does (SURVEY.md appendix C): registers placeholder modules for pyglet / gym / geometry /
duckietown_world / zuper_commons / carnivalmirror in ``sys.modules`` so that
``gym_duckietown.simulator``, ``.collision``, ``.graphics``, ``.distortion``,
``.envs.duckietown_env`` import, then builds a reference ``Simulator`` with ``object.__new__``
(skipping the GL-creating ``__init__``) and fills it through the reference's own ``_set_tile`` /
``_get_curve`` / ``WorldObj`` code.  Everything the returned object computes afterwards
(tile lookup, lane pose, reward, SAT collision, safety circles, done/reward, reset()'s RNG draw
order, fisheye LUT) is reference code executing, not a restatement.

What is NOT reference code here and therefore stays "parity unpinned":
  * duckietown_world dynamics (``get_DB18_nominal`` ...)       -> FakeDynamics below only records
    the initial pose; it never integrates.
  * duckietown_world ``get_transform`` (object placement)      -> ``_get_transform`` restates the
    README semantics (pos * tile_size -> (x, z), rotate in degrees about +y).
  * meshes / textures                                          -> extents come from the stand-in
    assets of the product package (same numbers on both sides).
"""
from __future__ import annotations

import importlib
import math
import os
import sys
import types
from unittest import mock

import numpy as np

REFERENCE_SRC = "/root/reference/src"


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_SRC, "gym_duckietown"))


class _Mock(types.ModuleType):
    """Module whose unknown attributes are MagicMocks (GL calls become no-ops)."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        m = mock.MagicMock(name=f"{self.__name__}.{name}")
        setattr(self, name, m)
        return m


class _SE2Transform:
    def __init__(self, p, theta):
        self.p = np.array(p, dtype=float)
        self.theta = float(theta)

    def as_SE2(self):
        c, s = math.cos(self.theta), math.sin(self.theta)
        return np.array([[c, -s, self.p[0]], [s, c, self.p[1]], [0.0, 0.0, 1.0]])


def _get_transform(desc, tm_h, tile_size):
    """README semantics of map objects (README.md:239); the real duckietown_world source is absent.

    The reference passes ``grid_width`` where the map HEIGHT is expected (simulator.py:936-938,
    SURVEY appendix B-8); this stand-in receives the sim through a global so it can undo that and
    always place ``pos=[px, pz]`` at world ``(px*ts, pz*ts)`` with ``angle = +rotate``.
    """
    px, pz = float(desc["pos"][0]), float(desc["pos"][1])
    gh = _get_transform.grid_height
    x = px * tile_size
    y = (gh - pz) * tile_size  # cartesian y so that weird z = pz * ts (simulator.py:1651)
    return _SE2Transform([x, y], math.radians(float(desc.get("rotate", 0.0))))


_get_transform.grid_height = 0


class FakeDynamics:
    """Placeholder for duckietown_world's PlatformDynamics: remembers c0, never integrates."""

    def __init__(self, **kw):
        self.kw = kw
        self.c0 = None

    def initialize(self, c0, t0=0, seed=None):
        self.c0 = c0
        return self


def _np_random(seed=None):
    """gym>=0.21 ``seeding.np_random``: Generator(PCG64(SeedSequence(seed)))."""
    ss = np.random.SeedSequence(seed)
    return np.random.Generator(np.random.PCG64(ss)), ss.entropy


_installed = False


def install():
    """Inject the stub modules and make ``gym_duckietown`` importable.  Idempotent."""
    global _installed
    if _installed:
        return
    if not reference_available():
        raise RuntimeError("reference tree not present at " + REFERENCE_SRC)
    names = [
        "pyglet", "pyglet.gl", "pyglet.image", "pyglet.window", "pyglet.graphics", "pyglet.text",
        "gym", "gym.spaces", "gym.utils", "gym.utils.seeding", "gym.envs", "gym.envs.registration",
        "geometry", "duckietown_world", "duckietown_world.resources", "duckietown_world.gltf",
        "duckietown_world.gltf.export", "duckietown_world.world_duckietown",
        "duckietown_world.world_duckietown.map_loading", "zuper_commons", "zuper_commons.logs",
        "zuper_commons.types", "carnivalmirror",
    ]
    mods = {}
    for n in names:
        m = _Mock(n)
        m.__path__ = []  # behave as a package
        mods[n] = m
        sys.modules[n] = m
    for n, m in mods.items():
        if "." in n:
            parent, child = n.rsplit(".", 1)
            setattr(mods[parent], child, m)

    gym = mods["gym"]

    class Env:  # real base classes: used in ``class`` statements (simulator.py:188, wrappers.py)
        metadata = {}
        reward_range = (-float("inf"), float("inf"))

        @property
        def unwrapped(self):
            return self

    class Wrapper(Env):
        def __init__(self, env):
            self.env = env
            self.action_space = getattr(env, "action_space", None)
            self.observation_space = getattr(env, "observation_space", None)

        @property
        def unwrapped(self):
            return self.env.unwrapped

        def reset(self, **kw):
            return self.env.reset(**kw)

        def step(self, a):
            return self.env.step(a)

    class ObservationWrapper(Wrapper):
        def reset(self, **kw):
            return self.observation(self.env.reset(**kw))

        def step(self, a):
            o, r, d, i = self.env.step(a)
            return self.observation(o), r, d, i

    class ActionWrapper(Wrapper):
        def step(self, a):
            return self.env.step(self.action(a))

    class RewardWrapper(Wrapper):
        def step(self, a):
            o, r, d, i = self.env.step(a)
            return o, self.reward(r), d, i

    class Box:
        def __init__(self, low, high, shape=None, dtype=np.float32):
            # like gym.spaces.Box: scalar bounds are broadcast to `shape`
            self.shape = tuple(shape) if shape is not None else np.shape(low)
            self.dtype = dtype
            self.low = np.full(self.shape, low, dtype=dtype) if np.isscalar(low) or np.ndim(low) == 0 else np.asarray(low)
            self.high = np.full(self.shape, high, dtype=dtype) if np.isscalar(high) or np.ndim(high) == 0 else np.asarray(high)

    class Discrete:
        def __init__(self, n):
            self.n = n

    gym.Env, gym.Wrapper = Env, Wrapper
    gym.ObservationWrapper, gym.ActionWrapper, gym.RewardWrapper = ObservationWrapper, ActionWrapper, RewardWrapper
    mods["gym.spaces"].Box, mods["gym.spaces"].Discrete = Box, Discrete
    mods["gym.utils.seeding"].np_random = _np_random

    class ZException(Exception):
        def __init__(self, msg=None, **kw):
            super().__init__(msg)

    mods["zuper_commons.types"].ZException = ZException
    mods["duckietown_world.resources"].list_maps2 = lambda: {}
    mods["duckietown_world.world_duckietown.map_loading"].get_transform = _get_transform
    dw = mods["duckietown_world"]
    dw.get_DB18_nominal = lambda delay: FakeDynamics(delay=delay)
    dw.get_DB18_uncalibrated = lambda delay, trim=0: FakeDynamics(delay=delay, trim=trim)
    dw.get_texture_file = lambda name: [name]

    class _MF1C:
        KIND_DUCKIEBOT = "duckiebot"
        KIND_DUCKIE = "duckie"
        KIND_TRAFFICLIGHT = "trafficlight"
        KIND_CHECKERBOARD = "checkerboard"
        ObjectKind = str

    dw.MapFormat1Constants = _MF1C
    dw.MapFormat1 = dict
    dw.MapFormat1Object = dict
    dw.SE2Transform = _SE2Transform
    mods["pyglet"].options = {"debug_gl": False}

    geo = mods["geometry"]
    geo.T3value = np.ndarray
    geo.SE2value = np.ndarray

    def SE2_from_translation_angle(t, theta):
        c, s = math.cos(theta), math.sin(theta)
        return np.array([[c, -s, t[0]], [s, c, t[1]], [0.0, 0.0, 1.0]])

    def translation_angle_from_SE2(q):
        return np.array([q[0, 2], q[1, 2]]), math.atan2(q[1, 0], q[0, 0])

    def se2_from_linear_angular(lin, ang):
        return np.array([[0.0, -ang, lin[0]], [ang, 0.0, lin[1]], [0.0, 0.0, 0.0]])

    geo.SE2_from_translation_angle = SE2_from_translation_angle
    geo.translation_angle_from_SE2 = translation_angle_from_SE2
    geo.se2_from_linear_angular = se2_from_linear_angular

    if REFERENCE_SRC not in sys.path:
        sys.path.insert(0, REFERENCE_SRC)
    _installed = True


def modules():
    """Return (simulator, collision, graphics, objects) reference modules."""
    install()
    S = importlib.import_module("gym_duckietown.simulator")
    C = importlib.import_module("gym_duckietown.collision")
    G = importlib.import_module("gym_duckietown.graphics")
    O = importlib.import_module("gym_duckietown.objects")
    return S, C, G, O


class FakeMesh:
    """Carries only what WorldObj / interpret_object read from an ObjMesh (objmesh.py:230-232)."""

    def __init__(self, min_coords, max_coords):
        self.min_coords = np.asarray(min_coords, dtype=np.float32)
        self.max_coords = np.asarray(max_coords, dtype=np.float32)
        self.textures = [None]

    def render(self, segment=False):
        pass


def build_reference_sim(map_data: dict, mesh_extents: dict, *, domain_rand=False, max_steps=1500,
                        seed=None, dynamics_rand=False, accept_start_angle_deg=60,
                        robot_speed=1.2, user_tile_start=None, cls=None):
    """Construct a reference ``Simulator`` (or subclass) without GL, loaded with ``map_data``.

    ``mesh_extents``: kind -> (min_coords[3], max_coords[3]) of the stand-in mesh for that kind.
    The map is interpreted by the reference's own ``_interpret_map`` (simulator.py:788-879).
    """
    S, C, G, O = modules()
    from gym_duckietown.randomization import Randomizer

    cls = cls or S.Simulator
    sim = object.__new__(cls)
    # attributes Simulator.__init__ sets before _load_map (simulator.py:256-346)
    sim.enable_leds = False
    sim.seed_value = seed
    sim.seed(seed=seed)
    sim.num_tris_distractors = 12
    sim.color_ground = (0.15, 0.15, 0.15)
    sim.color_sky = list(S.BLUE_SKY)
    sim.full_transparency = False
    sim.max_steps = max_steps
    sim.draw_curve = False
    sim.draw_bbox = False
    sim.domain_rand = domain_rand
    sim.randomizer = Randomizer()
    sim.frame_rate = 30
    sim.delta_time = 1.0 / 30
    sim.frame_skip = 1
    sim.graphics = True
    sim.camera_width, sim.camera_height = 160, 120
    sim.robot_speed = robot_speed
    sim.accept_start_angle_deg = accept_start_angle_deg
    sim.distortion = False
    sim.camera_rand = False
    sim.undistort = False
    sim.dynamics_rand = dynamics_rand
    sim.user_tile_start = user_tile_start
    sim.style = "photos"
    sim.randomize_maps_on_reset = False
    sim.step_count = 0
    sim.timestamp = 0.0
    sim.speed = 0.0
    sim.last_action = np.array([0, 0])
    sim.wheelVels = np.array([0, 0])
    sim.map_name = "standin"

    mesh_cache = {}

    def fake_get_mesh(kind, segment=False, change_materials=None):
        # cached per kind like ObjMesh.get (objmesh.py:28-62): TrafficLightObj instances SHARE their mesh, and
        # with it the card texture they assign in step() (objects.py:453,462)
        key = (kind, repr(change_materials))
        if key not in mesh_cache:
            lo, hi = mesh_extents[kind]
            mesh_cache[key] = FakeMesh(lo, hi)
            mesh_cache[key].kind = kind
        return mesh_cache[key]

    _get_transform.grid_height = len(map_data["tiles"])
    with mock.patch.object(S, "get_mesh", fake_get_mesh), \
            mock.patch.object(S, "get_duckiebot_mesh",
                              lambda color: FakeMesh(*mesh_extents.get("duckiebot", ([0, 0, 0], [1, 1, 1])))):
        sim._interpret_map(map_data)
    # reset() needs these no-op GL-side collaborators (simulator.py:634-656, 760)
    sim.render_obs = lambda segment=False: np.zeros((sim.camera_height, sim.camera_width, 3), np.uint8)
    S.load_texture = lambda *a, **k: object()
    return sim
