"""The fused fisheye gather (dts_set_fisheye_lut; k_bin<true>, build_binrec with per-fine-bin source boxes,
k_raster<*, true>, k_raster_solo<true>) against the CPU raster oracle with the same LUT: every frame EQUAL to the
oracle's, at the camera shapes that select different code paths —
  k_bin with one warp (<= 128 coarse bins: 160x120, 84x84, 90x70) or four (320x240, 640x480),
  k_raster_solo on (packed u8 HWC, W % 4 == 0) or off (90x70, wrapper layouts),
  partial coarse bins at the right edge (W = 84, 90) and partial fine-bin rows at the bottom (H = 70, 84) —
with the real LUT, the identity LUT (the fused path must equal the plain one), and synthetic LUTs that send output
bins to source boxes the real LUT never produces (mirrored, shuffled, zoomed, shrunk, jittered, half-integer, holes)."""
import os

import numpy as np
import pytest

from test_gpu_render import compare

pytestmark = pytest.mark.gpu

THREADS = os.cpu_count() or 1


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


@pytest.fixture(autouse=True)
def _default_tile_mode():
    import oracle as orc
    orc.lib().orr_set_tile_mode(1)
    yield
    orc.lib().orr_set_tile_mode(1)


def make_env(name, N, W, H, **kw):
    from gym_duckietown_b200.batched_env import BatchedDuckietownEnv
    args = dict(camera_width=W, camera_height=H, domain_rand=False, distortion=True, seed=5)
    args.update(kw)
    return BatchedDuckietownEnv(N, name, **args)


def drivable_poses(md, n, seed):
    """n random cameras on drivable tiles (as in test_large_batch_exact_and_order_independent)."""
    rng = np.random.default_rng(seed)
    ts = md.tile_size
    cells = np.array(md.drivable_tiles)[rng.integers(len(md.drivable_tiles), size=n)]
    return (cells[:, 0] + rng.uniform(size=n)) * ts, (cells[:, 1] + rng.uniform(size=n)) * ts, rng.uniform(-np.pi, np.pi, size=n)


def prop_poses(md, seed=5):
    """Cameras 0.15 .. 2.5 m from the map's props, facing them (as in test_small_triangle_path_vs_oracle)."""
    rng = np.random.default_rng(seed)
    poses = []
    for o in md.objects:
        for d in (0.15, 0.3, 0.5, 0.8, 1.2, 1.8, 2.5):
            a = rng.uniform(-np.pi, np.pi)
            poses.append((o.pos[0] - d * np.cos(a), o.pos[2] + d * np.sin(a), a + rng.uniform(-0.25, 0.25)))
    P = np.array(poses[:96])
    return P[:, 0].copy(), P[:, 1].copy(), P[:, 2].copy()


def place(env, px, pz, ang):
    env.sim.reset(None, dict(pos_x=px, pos_z=pz, angle=ang, map_id=np.zeros(len(px), np.int32)), env._stream())


def render_twice(env, torch):
    """Two renders of the same state: the fisheye bin lists are built with atomics, nothing may depend on their order."""
    a = env.render_obs().clone()
    b = env.render_obs(out=torch.empty_like(a))
    env.check()
    assert torch.equal(a, b), "two renders of the same state differ"
    return a.cpu().numpy()


def oracle_batch(md, px, pz, ang, W, H, lut, eps=None, domain_rand=False):
    import oracle as orc
    eps = eps or [orc.default_episode() for _ in range(len(px))]
    return orc.OracleScene(md).render_batch(px, pz, ang, eps, W, H, domain_rand, lut, threads=THREADS)


def assert_exact(gpu, cpu, tag):
    mx, frac = compare(gpu, cpu, tag)
    assert mx == 0, f"{tag}: max diff {mx} LSB on {frac:.2e} of the channel values"


def numpy_gather(frames, rx, ry):
    """cv2.remap(INTER_NEAREST, BORDER_CONSTANT) of plain frames: rint (half to even), outside and non-finite -> 0."""
    H, W = rx.shape
    ok = (np.abs(rx) < 2.0 ** 31) & (np.abs(ry) < 2.0 ** 31)      # False for NaN and +-inf
    ix = np.where(ok, np.rint(np.where(ok, rx, 0)), -1).astype(np.int64)
    iy = np.where(ok, np.rint(np.where(ok, ry, 0)), -1).astype(np.int64)
    ok &= (ix >= 0) & (ix < W) & (iy >= 0) & (iy < H)
    out = np.zeros_like(frames)
    out[:, ok] = frames[:, iy[ok], ix[ok]]
    return out


# ------------------------------------------------------------------------------------------------ LUTs
def lut_identity(W, H):
    return tuple(np.meshgrid(np.arange(W, dtype=np.float32), np.arange(H, dtype=np.float32)))


def lut_mirror(W, H, rng):
    x, y = lut_identity(W, H)
    return W - 1 - x, H - 1 - y


def lut_bin_shuffle(W, H, rng):
    """Output coarse bin b reads the 32x8 source block of bin perm[b], shifted by (1..31, 1..7) px: every source box
    straddles two source cells in x and in y."""
    x, y = lut_identity(W, H)
    nx, ny = (W + 31) // 32, (H + 7) // 8
    perm = rng.permutation(nx * ny)
    dx, dy = rng.integers(1, 32, nx * ny), rng.integers(1, 8, nx * ny)
    b = (y.astype(int) // 8) * nx + x.astype(int) // 32
    p = perm[b]
    return ((p % nx) * 32 + x % 32 + dx[b]).astype(np.float32), ((p // nx) * 8 + y % 8 + dy[b]).astype(np.float32)


def lut_zoom2(W, H, rng):
    x, y = lut_identity(W, H)
    return x / 2, y / 2


def lut_shrink2(W, H, rng):
    x, y = lut_identity(W, H)
    return 2 * x, 2 * y


def lut_jitter(W, H, rng):
    x, y = lut_identity(W, H)
    return (x + rng.uniform(-3, 3, x.shape)).astype(np.float32), (y + rng.uniform(-3, 3, y.shape)).astype(np.float32)


def lut_ties(W, H, rng):
    """Exact halves: -0.5 rounds to 0 (inside), W - 0.5 to W (outside for even W)."""
    x, y = lut_identity(W, H)
    return x + np.float32(0.5), y - np.float32(0.5)


def lut_holes(W, H, rng):
    """The real LUT with scattered NaN, +-inf, +-1e9, +-3e9 entries, one whole fine bin and one whole coarse bin of NaN."""
    from gym_duckietown_b200.distortion import Distortion
    d = Distortion(W, H)
    rx, ry = d.rmapx.copy(), d.rmapy.copy()
    bad = np.array([np.nan, np.inf, -np.inf, 1e9, -1e9, 3e9, -3e9], np.float32)
    for tgt in (rx, ry):
        pick = rng.random(tgt.shape) < 0.02
        tgt[pick] = bad[rng.integers(len(bad), size=int(pick.sum()))]
    fx, fy = rng.integers(0, W // 8) * 8, rng.integers(0, H // 4) * 4
    rx[fy:fy + 4, fx:fx + 8] = np.nan
    cx, cy = rng.integers(0, W // 32) * 32, rng.integers(0, H // 8) * 8
    ry[cy:cy + 8, cx:cx + 32] = np.nan
    return rx, ry


SYNTH = dict(mirror=lut_mirror, bin_shuffle=lut_bin_shuffle, zoom2=lut_zoom2, shrink2=lut_shrink2, jitter=lut_jitter,
             ties=lut_ties, holes=lut_holes)


def widest_box(rx, ry):
    """The largest H*w + W*h over the coarse bins' source boxes: what dts_set_fisheye_lut holds against its int32 budget."""
    H, W = rx.shape
    ok = (np.abs(rx) < 2.0 ** 31) & (np.abs(ry) < 2.0 ** 31)
    sx = np.where(ok, np.rint(np.where(ok, rx, 0)), -1).astype(np.int64)
    sy = np.where(ok, np.rint(np.where(ok, ry, 0)), -1).astype(np.int64)
    ok &= (sx >= 0) & (sx < W) & (sy >= 0) & (sy < H)
    best = 0
    for y0 in range(0, H, 8):
        for x0 in range(0, W, 32):
            m = ok[y0:y0 + 8, x0:x0 + 32]
            if m.any():
                bx, by = sx[y0:y0 + 8, x0:x0 + 32][m], sy[y0:y0 + 8, x0:x0 + 32][m]
                best = max(best, H * int(bx.max() - bx.min() + 2) + W * int(by.max() - by.min() + 2))
    return best


# ------------------------------------------------------------------------------------------------ 1. real LUT, large batches
@pytest.mark.parametrize("name,W,H,N,poses,tess", [
    ("small_loop", 160, 120, 2048, "drivable", False), ("loop_obstacles", 160, 120, 2048, "drivable", False),
    ("loop_obstacles", 90, 70, 1024, "drivable", False), ("small_loop", 84, 84, 1024, "drivable", False),
    ("udem1", 320, 240, 512, "drivable", False), ("udem1", 640, 480, 256, "drivable", False),
    ("loop_obstacles", 160, 120, 96, "props", False), ("loop_obstacles", 160, 120, 1024, "drivable", True)])
def test_real_lut_large_batch_exact_and_order_independent(name, W, H, N, poses, tess, torch_cuda):
    """Random cameras (or cameras facing the props: sub-pixel prop triangles, which take the warp path under fisheye)
    through the reference LUT: every frame equal to the oracle's, two renders equal to each other."""
    import oracle as orc
    from gym_duckietown_b200 import maps
    md = maps.load_map(name)
    px, pz, ang = prop_poses(md) if poses == "props" else drivable_poses(md, N, 2024 + W)
    orc.lib().orr_set_tile_mode(0 if tess else 1)
    env = make_env(name, len(px), W, H, tessellate_tiles=tess)
    place(env, px, pz, ang)
    gpu = render_twice(env, torch_cuda)
    cpu = oracle_batch(md, px, pz, ang, W, H, (env.camera_model.rmapx, env.camera_model.rmapy))
    assert_exact(gpu, cpu, f"fish_real_{name}_{W}x{H}_{poses}{'_tess' if tess else ''}")
    assert gpu.std() > 10
    env.close()


# ------------------------------------------------------------------------------------------------ 2. episodes
@pytest.mark.parametrize("name,W,H,N", [("loop_obstacles", 160, 120, 64), ("udem1", 160, 120, 64), ("udem1", 640, 480, 8)])
def test_episodes_with_device_resets_vs_oracle(name, W, H, N, torch_cuda):
    """domain_rand + device auto-reset under fisheye: drive until some envs have started a new episode (DR camera,
    lighting, hidden objects, the stale light of second episodes), then compare the last observation with the oracle
    driven by the product's episode records."""
    torch = torch_cuda
    import oracle as orc
    from gym_duckietown_b200 import maps
    env = make_env(name, N, W, H, domain_rand=True, seed=60, device_reset=True, auto_reset=True)
    env.reset()
    g = torch.Generator().manual_seed(7)
    acts = torch.stack([torch.full((N,), 1.0), torch.rand(N, generator=g) * 1.2 - 0.6], 1).to(env.device)
    for t in range(160):
        obs, _, _, info = env.step(acts)
        if t >= 39 and int(info["episode"].max()) > 1:
            break
    env.check()
    st = {k: v.cpu().numpy() for k, v in info.items()}
    assert st["episode"].max() > 1, "no env reset"
    eps = []
    for k in range(N):
        r = env.sim.debug_episode(k)
        eps.append(orc.default_episode(cam_height=float(r["cam_height"]), cam_angle_deg=float(r["cam_angle_deg"]),
                                       cam_fov_y_deg=float(r["cam_fov_y_deg"]), cam_noise=r["cam_noise"], horizon=r["horizon"],
                                       ambient=r["ambient"], diffuse=r["diffuse"], light_eye=r["light_eye"], ground=r["ground"],
                                       hidden=[int(v) for v in r["hidden"]]))
    cpu = oracle_batch(maps.load_map(name), st["pos_x"], st["pos_z"], st["angle"], W, H,
                       (env.camera_model.rmapx, env.camera_model.rmapy), eps, domain_rand=True)
    assert_exact(obs.cpu().numpy(), cpu, f"fish_episodes_{name}_{W}x{H}")
    env.close()


# ------------------------------------------------------------------------------------------------ 3. identity LUT
@pytest.mark.parametrize("name,W,H,variant", [
    ("loop_obstacles", 160, 120, "plain"), ("udem1", 160, 120, "plain"), ("loop_obstacles", 640, 480, "plain"),
    ("udem1", 640, 480, "plain"), ("udem1", 160, 120, "segment"), ("loop_obstacles", 160, 120, "tess"),
    ("loop_obstacles", 160, 120, "cwh_u8")])
def test_identity_lut_equals_plain_path(name, W, H, variant, torch_cuda):
    """With the identity LUT the fused path (source boxes, inverse indices, fine-bin accept bits against boxes, no
    one-lane-per-triangle path) must produce exactly what the plain path produces, 2048 cameras at a time."""
    torch = torch_cuda
    from gym_duckietown_b200 import maps
    N = 2048
    px, pz, ang = drivable_poses(maps.load_map(name), N, 99 + W)
    kw = dict(tessellate_tiles=variant == "tess")
    fish, plain = make_env(name, N, W, H, **kw), make_env(name, N, W, H, distortion=False, **kw)
    fish.sim.set_fisheye_lut(*lut_identity(W, H))
    got = []
    for env in (fish, plain):
        if variant == "cwh_u8":
            env.set_output_format(obs_layout="cwh", obs_dtype="uint8")
        place(env, px, pz, ang)
        got.append(env.render_obs(segment=variant == "segment").clone())
        env.check()
    assert torch.equal(got[0], got[1]), f"{int((got[0] != got[1]).sum())} channel values differ"
    assert float(got[1][:64].float().std()) > 10
    fish.close(); plain.close()


# ------------------------------------------------------------------------------------------------ 4. synthetic LUTs
@pytest.mark.parametrize("W,H,N", [(160, 120, 256), (90, 70, 256), (640, 480, 32)])
@pytest.mark.parametrize("lut", list(SYNTH))
def test_synthetic_lut_vs_oracle(lut, W, H, N, torch_cuda):
    """Source boxes in other cells than their output bins (mirror), straddling cells (bin_shuffle), shared by many bins
    (zoom2), empty or partly empty (shrink2, holes), overlapping (jitter), exact halves (ties): equal to the oracle with
    the same LUT, and the oracle equal to a numpy gather of its plain frames."""
    from gym_duckietown_b200 import maps
    name = "udem1" if W == 640 else "loop_obstacles"
    md = maps.load_map(name)
    rx, ry = SYNTH[lut](W, H, np.random.default_rng(W + len(lut)))
    env = make_env(name, N, W, H)
    real = widest_box(env.camera_model.rmapx, env.camera_model.rmapy)
    assert widest_box(rx, ry) <= 1.5 * real
    env.sim.set_fisheye_lut(rx, ry)
    px, pz, ang = drivable_poses(md, N, 31 + W)
    place(env, px, pz, ang)
    gpu = render_twice(env, torch_cuda)
    cpu = oracle_batch(md, px, pz, ang, W, H, (rx, ry))
    flat = oracle_batch(md, px[:8], pz[:8], ang[:8], W, H, None)
    assert np.array_equal(cpu[:8], numpy_gather(flat, rx, ry))
    assert_exact(gpu, cpu, f"fish_{lut}_{W}x{H}")
    if lut in ("shrink2", "holes", "ties"):
        assert (gpu == 0).all(-1).any(-1).any(-1).all()   # pixels sent outside the image are black
    env.close()


# ------------------------------------------------------------------------------------------------ 5. replacing / refusing
def test_replacing_and_refusing_a_lut(torch_cuda):
    """Setting a LUT replaces every table built from the previous one; a LUT the rasteriser cannot take (a source box
    too wide for its int32 edge functions, the wrong size) is refused and the previous one stays in effect."""
    torch = torch_cuda
    from gym_duckietown_b200 import lib as L, maps
    N, W, H = 4, 640, 480
    env = make_env("udem1", N, W, H)
    place(env, *drivable_poses(maps.load_map("udem1"), N, 3))
    a = env.render_obs().clone()
    rng = np.random.default_rng(4)
    env.sim.set_fisheye_lut(*lut_bin_shuffle(W, H, rng))
    b = env.render_obs().clone()
    assert not torch.equal(a, b)
    env.sim.set_fisheye_lut(env.camera_model.rmapx, env.camera_model.rmapy)
    assert torch.equal(env.render_obs().clone(), a)
    # output bin 27 (row 1, column 7 of the 20 x 60 coarse bins) scattered over the whole source image
    wide = [v.copy() for v in lut_identity(W, H)]
    wide[0][8:16, 224:256] = rng.uniform(0, W - 1, (8, 32)).astype(np.float32)
    wide[1][8:16, 224:256] = rng.uniform(0, H - 1, (8, 32)).astype(np.float32)
    wide[0][8, 224], wide[1][8, 224], wide[0][15, 255], wide[1][15, 255] = 0, 0, W - 1, H - 1
    with pytest.raises(L.DtsError, match="output bin 27 "):
        env.sim.set_fisheye_lut(*wide)
    with pytest.raises(L.DtsError, match="is 320x240 but the camera is 640x480"):
        env.sim.set_fisheye_lut(*lut_identity(320, 240))
    assert torch.equal(env.render_obs().clone(), a)
    env.check()
    env.close()


# ------------------------------------------------------------------------------------------------ 6. other fused features
@pytest.mark.parametrize("W,H", [(90, 70), (160, 120)])
def test_fisheye_wrapper_layouts_vs_oracle(W, H, torch_cuda):
    """Fisheye with ImgWrapper / PyTorchObsWrapper layouts and NormalizeWrapper's /255 fused in (k_raster<true, true>,
    no solo kernel, the planar u8 edge stores)."""
    from gym_duckietown_b200 import maps
    N = 64
    md = maps.load_map("udem1")
    env = make_env("udem1", N, W, H)
    px, pz, ang = drivable_poses(md, N, 8)
    place(env, px, pz, ang)
    ref = oracle_batch(md, px, pz, ang, W, H, (env.camera_model.rmapx, env.camera_model.rmapy))
    for layout, perm in (("chw", (0, 3, 1, 2)), ("cwh", (0, 3, 2, 1))):
        for dtype in ("uint8", "float32"):
            env.set_output_format(obs_layout=layout, obs_dtype=dtype)
            got = env.render_obs().cpu().numpy()
            env.check()
            want = ref.transpose(perm)
            if dtype == "float32":
                assert got.dtype == np.float32 and np.array_equal(got, (want / 255.0).astype(np.float32)), (layout, dtype)
            else:
                assert_exact(got.transpose(np.argsort(perm)), ref, f"fish_layout_{layout}_{W}x{H}")
    env.close()


def test_fisheye_resize_equals_resize_of_fisheye_frames(torch_cuda):
    """ResizeWrapper fused behind the fisheye gather equals the device resize applied to the fisheye frames."""
    torch = torch_cuda
    from gym_duckietown_b200 import maps
    N, W, H = 64, 160, 120
    md = maps.load_map("loop_obstacles")
    env = make_env("loop_obstacles", N, W, H)
    px, pz, ang = drivable_poses(md, N, 12)
    place(env, px, pz, ang)
    frames = env.render_obs().clone()
    assert_exact(frames.cpu().numpy(), oracle_batch(md, px, pz, ang, W, H, (env.camera_model.rmapx, env.camera_model.rmapy)),
                 "fish_resize_frames")
    env.set_resize(84, 84)
    fused = env.render_obs().clone()
    assert fused.shape == (N, 84, 84, 3)
    assert torch.equal(fused, env.sim_resize_only(frames).clone())
    env.check()
    env.close()


@pytest.mark.parametrize("W,H,N", [(640, 480, 8), (90, 70, 64)])
def test_fisheye_fused_gather_vs_oracle(W, H, N, torch_cuda):
    """FusedObsGather under fisheye: at 640x480 most coarse bins are drawn by k_raster_solo, and the row blocks drawn
    entirely by it must still reach the gather buffer."""
    torch = torch_cuda
    from gym_duckietown_b200 import maps
    from gym_duckietown_b200.dist import FusedObsGather
    md = maps.load_map("udem1")
    env = make_env("udem1", N, W, H)
    px, pz, ang = drivable_poses(md, N, 21)
    place(env, px, pz, ang)
    g = FusedObsGather(env, 0, 1)
    g.arm()
    obs = env.render_obs()
    out = g.finish()
    env.check()
    assert torch.equal(out[0], obs)
    assert_exact(obs.cpu().numpy(), oracle_batch(md, px, pz, ang, W, H, (env.camera_model.rmapx, env.camera_model.rmapy)),
                 f"fish_gather_{W}x{H}")
    env.close()


@pytest.mark.parametrize("name", ["loop_obstacles", "udem1"])
def test_fisheye_segment_view_vs_oracle(name, torch_cuda):
    """render_obs(segment=True) is distorted too (the reference's render_obs applies the camera model to it)."""
    import oracle as orc
    from gym_duckietown_b200 import maps
    N, W, H = 24, 160, 120
    md = maps.load_map(name)
    env = make_env(name, N, W, H)
    px, pz, ang = drivable_poses(md, N, 17)
    place(env, px, pz, ang)
    got = env.render_obs(segment=True).cpu().numpy()
    env.check()
    sc = orc.OracleScene(md)
    lut = (env.camera_model.rmapx, env.camera_model.rmapy)
    ref = np.stack([sc.render(px[k], pz[k], ang[k], None, W, H, lut=lut, segment=True) for k in range(N)])
    assert_exact(got, ref, f"fish_segment_{name}")
    assert (got == np.array([255, 0, 255], np.uint8)).all(-1).mean() > 0.05
    env.close()
