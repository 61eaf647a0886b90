"""SURVEY 8f-3 / boundary: the fused wrapper path against the reference's OWN wrapper classes.

tests/golden/wrappers.npz was produced by running src/gym_duckietown/wrappers.py and learning/utils/wrappers.py
unmodified (stub-imported, oracle/make_golden.py gen_wrappers) on canned frames / rewards / actions.  CPU part:
the numpy semantics the GPU tests rely on are those outputs.  GPU part (-m gpu): the device ResizeWrapper
(dts_set_resize) against cv2.INTER_CUBIC as the reference wrapper called it."""
import hashlib
import os

import numpy as np
import pytest

from gym_duckietown_b200.gymshim import spaces
from gym_duckietown_b200.simulator import Simulator

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "wrappers.npz")
GOLD_INTERFACE = os.path.join(ROOT, "tests", "golden", "wrapper_interface.npz")


def canned_frames(seed, h, w):
    """Same draws as gen_wrappers (one rng, 160x120 first then 640x480)."""
    rng = np.random.default_rng(seed)
    out = {}
    for tag, (hh, ww) in {"160x120": (120, 160), "640x480": (480, 640)}.items():
        frames = rng.integers(0, 256, (3, hh, ww, 3), dtype=np.uint8)
        yy, xx = np.mgrid[0:hh, 0:ww]
        frames[2] = np.stack([(xx * 255 // ww), (yy * 255 // hh), ((xx + yy) * 255 // (hh + ww))], -1).astype(np.uint8)
        out[tag] = frames
    return out[f"{w}x{h}"]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.parametrize("tag", ["160x120", "640x480"])
def test_observation_wrapper_semantics_are_the_reference_classes(tag):
    g = np.load(GOLD)
    w, h = map(int, tag.split("x"))
    frames = canned_frames(int(g["seed"]), h, w)
    assert sha(frames) == str(g[f"frames_sha_{tag}"])
    assert sha(np.stack([f.transpose(2, 1, 0) for f in frames])) == str(g[f"pytorch_sha_{tag}"])     # PyTorchObsWrapper W:110
    assert sha(np.stack([f.transpose(2, 0, 1) for f in frames])) == str(g[f"img_sha_{tag}"])         # ImgWrapper LW:86
    assert sha((frames[:1] / 255.0).astype(np.float32)) == str(g[f"norm_f32_sha_{tag}"])            # NormalizeWrapper LW:66-70
    assert str(g[f"norm_dtype_{tag}"]) == "float64"


def test_reward_and_action_wrapper_semantics_are_the_reference_classes():
    g = np.load(GOLD)
    r = g["rewards"]
    assert np.array_equal(g["dt_rewards"], np.where(r == -1000, -10.0, np.where(r > 0, r + 10, r + 4)))   # DtRewardWrapper LW:94-102
    assert np.array_equal(g["scaled_actions"], g["actions"] * [0.8, 1.0])                                # ActionWrapper LW:110-112
    assert np.array_equal(g["discrete_actions"], [[0.6, 1.0], [0.6, -1.0], [0.7, 0.0]])                   # DiscreteWrapper W:18-30


class StandIn:
    """The attributes gym_duckietown_b200.Simulator.__init__ sets (simulator.py) and its step / reset signature, without
    CUDA: what a wrapper of the reference sees of the product env."""
    metadata, reward_range = Simulator.metadata, (-1000, 1000)
    action_space = spaces.Box(low=-1, high=1, shape=(2,), dtype=np.float32)
    observation_space = spaces.Box(low=0, high=255, shape=(120, 160, 3), dtype=np.uint8)

    @property
    def unwrapped(self):
        return self

    def reset(self):
        return np.zeros((120, 160, 3), np.uint8)

    def step(self, a):
        return np.ones((120, 160, 3), np.uint8), 0.0, False, {}


def test_unmodified_reference_wrappers_accept_the_product_env_interface():
    """The reference's wrappers.py, imported unmodified, wrapped StandIn in PyTorchObsWrapper and ResizeWrapper(84, 84)
    as the PyTorchObsWrapper block of run_tests.py:28-34 does; tests/golden/wrapper_interface.npz holds the spaces and
    shapes they returned.  StandIn must still offer what those wrappers read (W:96-103, 112-120: the observation
    space's shape, dtype, low[0, 0, 0], high[0, 0, 0], high[1, 1, 1]; reset() and a 4-tuple step()) with the values
    recorded, and the product's fused wrappers must declare the same spaces."""
    from gym_duckietown_b200 import wrappers as PW
    from gym_duckietown_b200.batched_env import BatchedDuckietownEnv
    g = np.load(GOLD_INTERFACE)
    env = StandIn()
    sp = env.observation_space
    assert [sp.shape[2], sp.shape[1], sp.shape[0]] == g["pytorch_shape"].tolist()
    assert np.dtype(sp.dtype).str == str(g["pytorch_dtype"]) == str(g["resize_dtype"])
    assert sp.low[0, 0, 0] == g["pytorch_low"][0] == g["resize_low"][0]
    assert sp.high[0, 0, 0] == g["pytorch_high"][0] and sp.high[1, 1, 1] == g["resize_high"][0]
    first, (second, _, _, _) = env.reset(), env.step([0, 0])
    assert [first.T.shape, second.T.shape] == [tuple(s) for s in g["obs_shapes"]]      # observation(): transpose(2, 1, 0)
    assert g["resize_shape"].tolist() == g["resize_reset_shape"].tolist() == [3, 84, 84]

    class Batched:   # the part of BatchedDuckietownEnv the fused wrappers configure
        camera_width, camera_height, resize = 160, 120, None
        obs_size = BatchedDuckietownEnv.obs_size

        def __init__(self):
            self.output_format = dict(obs_layout="hwc", obs_dtype="uint8")

        def set_output_format(self, obs_layout=None, obs_dtype=None, **kw):
            self.output_format.update({k: v for k, v in (("obs_layout", obs_layout), ("obs_dtype", obs_dtype)) if v})

        def set_resize(self, w, h):
            self.resize = (w, h)

    pt = PW.PyTorchObsWrapper(Batched())
    rz = PW.ResizeWrapper(PW.PyTorchObsWrapper(Batched()), resize_w=84, resize_h=84)
    for tag, space in (("pytorch", pt.observation_space), ("resize", rz.observation_space)):
        assert list(space.shape) == g[f"{tag}_shape"].tolist(), tag
        assert np.dtype(space.dtype).str == str(g[f"{tag}_dtype"]), tag
        assert space.low.flat[0] == g[f"{tag}_low"][0] and space.high.flat[0] == g[f"{tag}_high"][0], tag


@pytest.mark.gpu
@pytest.mark.parametrize("tag,rw,rh", [("160x120", 84, 84), ("160x120", 80, 80), ("160x120", 64, 48), ("640x480", 84, 84)])
def test_device_resize_vs_reference_resize_wrapper(tag, rw, rh):
    """dts_set_resize vs the frames the reference's ResizeWrapper(PyTorchObsWrapper(env)) returned (cv2.INTER_CUBIC):
    <= 1 LSB everywhere (OpenCV's vector path and the fixed-point restatement round a few percent of the values
    differently), and exact agreement of the restatement with itself across layouts."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from gym_duckietown_b200.batched_env import BatchedDuckietownEnv
    g = np.load(GOLD)
    w, h = map(int, tag.split("x"))
    frames = canned_frames(int(g["seed"]), h, w)
    want = g[f"resize_{tag}_{rw}x{rh}"]                    # [3][C][rw][rh]
    env = BatchedDuckietownEnv(3, "small_loop", camera_width=w, camera_height=h, domain_rand=False, seed=1)
    env.reset(render=False)
    env.set_output_format(obs_layout="cwh")
    env.set_resize(rw, rh)
    assert tuple(env.obs.shape) == (3, 3, rw, rh)
    src = torch.from_numpy(frames).to(env.device)
    got = env.sim_resize_only(src).cpu().numpy()
    d = np.abs(got.astype(int) - want.astype(int))
    assert d.max() <= 1, d.max()
    assert (d > 0).mean() < 0.08
    env.set_output_format(obs_layout="hwc")
    hwc = env.sim_resize_only(src).cpu().numpy()
    assert np.array_equal(hwc.transpose(0, 3, 2, 1), got)
    # the tiled kernel (bands of output rows staged in shared memory) against the one-thread-per-pixel kernel: same integers
    import os
    os.environ["DTS_RESIZE_UNTILED"] = "1"
    try:
        env.set_resize(rw, rh)
        assert np.array_equal(env.sim_resize_only(src).cpu().numpy(), hwc)
        env.set_output_format(obs_layout="chw", obs_dtype="float32")
        untiled_f32 = env.sim_resize_only(src).cpu().numpy()
    finally:
        del os.environ["DTS_RESIZE_UNTILED"]
    env.set_resize(rw, rh)
    assert np.array_equal(env.sim_resize_only(src).cpu().numpy(), untiled_f32)
    env.close()
