"""The reference's own smoke script (run_tests.py:10-52) replayed against the drop-in classes, plus
fisheye / MultiMap / auto-reset behaviour through the public API."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def test_run_tests_script_equivalent(torch_cuda):
    from gym_duckietown_b200 import gymshim
    from gym_duckietown_b200.simulator import DuckietownEnv, MultiMapEnv

    env = gymshim.make("Duckietown-udem1-v0", camera_width=160, camera_height=120)   # run_tests.py:10
    env.reset()
    for _ in range(10):
        obs, _, _, _ = env.step(np.array([0.1, 0.1]))                                # :13-14
    first_obs = env.reset()
    first_render = env.render("rgb_array")                                           # :17-22
    m0, m1 = first_obs.mean(), first_render.mean()
    assert 0 < m0 < 255 and abs(m0 - m1) < 5
    second_obs, rew, done, info = env.step([0.0, 0.0])                               # :25-27
    assert first_obs.shape == env.observation_space.shape == second_obs.shape
    assert first_obs.dtype == np.uint8 and isinstance(rew, float) and isinstance(done, bool)
    assert "Simulator" in info and "DuckietownEnv" in info and "action" in info["Simulator"]
    assert first_render.shape == (600, 800, 3)                                       # WINDOW_HEIGHT x WINDOW_WIDTH S:100-101
    top = env.render("top_down")
    seg = env.render_obs(segment=True)
    # (the env is unseeded like the reference's script: which class shows in a given pixel varies from run to run, so
    # only ask that the clear / ground colour of segment mode, magenta, is on screen)
    assert top.shape == (600, 800, 3) and top.std() > 5 and seg.shape == first_obs.shape
    assert (seg == np.array([255, 0, 255], np.uint8)).all(-1).mean() > 0.05
    assert env.reset(segment=True).shape == first_obs.shape
    from gym_duckietown_b200.wrappers import PyTorchObsWrapper                       # :28-34
    env = PyTorchObsWrapper(env)
    first_obs = env.reset()
    second_obs, _, _, _ = env.step([0, 0])
    assert first_obs.shape == tuple(env.observation_space.shape) == second_obs.shape == (3, 160, 120)
    env.close()
    for map_name in ["loop_only_duckies", "small_loop_only_duckies"]:               # :37-39
        e = DuckietownEnv(map_name=map_name, camera_width=84, camera_height=84)
        e.reset()
        e.close()
    mm = MultiMapEnv(camera_width=84, camera_height=84)                              # :42-44
    seen = set()
    for _ in range(6):
        mm.reset()
        seen.add(mm.cur_env_idx)
    assert seen == {0, 1}
    mm.close()
    env = DuckietownEnv(map_name="loop_obstacles", camera_width=84, camera_height=84)   # :47-52
    for _ in range(75):
        env.reset()
        assert not env._collision_at(env.cur_pos, env.cur_angle), "collision on spawn"
        env.step(np.array([0.05, 0]))
        assert not env._collision_at(env.cur_pos, env.cur_angle), "collision after one step"
    env.close()


def test_full_transparency_info_and_helpers(torch_cuda):
    from gym_duckietown_b200.simulator import DuckietownEnv, NotInLane
    env = DuckietownEnv(map_name="small_loop", domain_rand=False, camera_width=84, camera_height=84,
                        full_transparency=True, seed=3)
    _, _, _, info = env.step([0.3, 0.0])
    s = info["Simulator"]
    for key in ("lane_position", "robot_speed", "proximity_penalty", "cur_pos", "cur_angle", "wheel_velocities",
                "timestamp", "tile_coords"):
        assert key in s
    lp = env.get_lane_pos2(env.cur_pos, env.cur_angle)
    assert abs(lp.dist - s["lane_position"]["dist"]) < 1e-12
    assert env.get_grid_coords(env.cur_pos) == tuple(s["tile_coords"])
    with pytest.raises(NotInLane):
        env.get_lane_pos2(np.array([0.1, 0, 0.1]), 0.0)   # grass tile
    assert env._valid_pose(env.cur_pos, env.cur_angle)
    env.close()


def test_fisheye_fused_gather_vs_oracle(torch_cuda):
    """config 4 shape: 640x480 + distortion (+ domain_rand): the fused gather equals rendering the
    undistorted frame with the oracle and applying the reference LUT."""
    torch = torch_cuda
    import oracle as orc
    from gym_duckietown_b200 import maps
    from gym_duckietown_b200.batched_env import BatchedDuckietownEnv
    from test_gpu_render import oracle_episode

    N, W, H = 6, 640, 480
    env = BatchedDuckietownEnv(N, "udem1", camera_width=W, camera_height=H, domain_rand=True, distortion=True, seed=50)
    captured = {}
    orig = env.sim.reset
    env.sim.reset = lambda mask, params, stream=0: (captured.update(params), orig(mask, params, stream))[1]
    obs = env.reset()
    torch.cuda.synchronize()
    st = {k: v.cpu().numpy() for k, v in env.state.items()}
    sc = orc.OracleScene(maps.load_map("udem1"))
    lut = (env.camera_model.rmapx, env.camera_model.rmapy)
    gpu = obs.cpu().numpy()
    for k in range(N):
        cpu = sc.render(st["pos_x"][k], st["pos_z"][k], st["angle"][k], oracle_episode(orc, captured, k), W, H, True, lut)
        undist = sc.render(st["pos_x"][k], st["pos_z"][k], st["angle"][k], oracle_episode(orc, captured, k), W, H, True)
        assert np.array_equal(env.camera_model.distort(undist), cpu)   # oracle gather == product's numpy gather
        d = np.abs(gpu[k].astype(int) - cpu.astype(int))
        assert d.max() == 0, (k, d.max(), int((d > 0).sum()))
    env.check()
    env.close()


def test_multimap_cycle_and_stale_light_on_device(torch_cuda):
    """config 5 semantics: map id advances on every reset (device-side); second episodes capture the
    light under the previous frame's modelview (S:581)."""
    torch = torch_cuda
    from gym_duckietown_b200.batched_env import BatchedDuckietownEnv
    env = BatchedDuckietownEnv(256, ["loop_only_duckies", "small_loop_only_duckies"], camera_width=84, camera_height=84,
                               domain_rand=False, seed=5, auto_reset=True, device_reset=True, cycle_maps=True)
    env.reset()
    torch.cuda.synchronize()
    assert (env.state["map_id"] == 0).all()
    env.reset()
    torch.cuda.synchronize()
    assert (env.state["map_id"] == 1).all()
    acts = torch.zeros((256, 2), device=env.device)
    acts[:, 0] = 1.0
    acts[:, 1] = 1.0
    for _ in range(120):
        obs, rew, done, info = env.step(acts)
    torch.cuda.synchronize()
    ep = info["episode"].cpu().numpy()
    mid = info["map_id"].cpu().numpy()
    assert ((ep - 1) % 2 == mid).all() and ep.max() > 2
    assert obs.float().std() > 5
    env.close()


def test_host_pipeline_matches_sequential_stepping(torch_cuda):
    """HostPipeline (double-buffered H2D / D2H) returns exactly what step-by-step device stepping returns."""
    torch = torch_cuda
    from gym_duckietown_b200.batched_env import BatchedDuckietownEnv, HostPipeline
    kw = dict(camera_width=84, camera_height=84, domain_rand=False, seed=11, auto_reset=True, device_reset=True)
    a, b = BatchedDuckietownEnv(300, "loop_obstacles", **kw), BatchedDuckietownEnv(300, "loop_obstacles", **kw)
    a.reset(); b.reset()
    acts = torch.empty((12, 300, 2)).uniform_(-1, 1).pin_memory()
    pipe = HostPipeline(b, depth=2)
    tickets = []
    for t in range(12):
        tickets.append(pipe.submit(acts[t]))
        if t >= 1:
            ho, hr, hd = pipe.result(tickets[t - 1])
            assert np.array_equal(ho.numpy(), ref[0]) and np.array_equal(hr.numpy(), ref[1]) and np.array_equal(hd.numpy(), ref[2])
        o, r, d, _ = a.step(acts[t].to(a.device))
        torch.cuda.synchronize()
        ref = (o.cpu().numpy().copy(), r.cpu().numpy().copy(), d.cpu().numpy().copy())
    ho, hr, hd = pipe.result(tickets[-1])
    assert np.array_equal(ho.numpy(), ref[0]) and np.array_equal(hd.numpy(), ref[2])
    a.close(); b.close()


def test_simulator_randomize_maps_on_reset(torch_cuda):
    """Simulator(randomize_maps_on_reset=True) (S:373-378, 541-544): the map changes between resets and the
    map-dependent attributes follow it."""
    import gym_duckietown_b200 as gd
    env = gd.Simulator("small_loop", randomize_maps_on_reset=True, camera_width=84, camera_height=84, seed=3, domain_rand=False)
    names = set()
    for _ in range(8):
        obs = env.reset()
        assert obs.shape == (84, 84, 3)
        names.add(env.map_name)
        md = gd.maps.load_map(env.map_name)
        assert (env.grid_width, env.grid_height) == (md.grid_w, md.grid_h)
        i, j = env.get_grid_coords(env.cur_pos)
        assert md.tile_drivable[j * md.grid_w + i]
        env.step([0.3, 0.3])
    assert len(names) >= 3
    env.close()
