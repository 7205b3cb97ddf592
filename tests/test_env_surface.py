"""The reference's class surface (gym.Env reset/step, AssistiveEnv / Agent / Robot / Human) on the
batched backend: shapes, spaces, and agreement between the fused step and the same step done through
the reference-shaped per-call API (take_step + _get_obs + get_food_rewards + human_preferences)."""
import numpy as np
import pytest

from assistive_gym_b200 import capi


def _make(lib, n_envs, seed):
    from assistive_gym_b200 import envs
    env = envs.make('assistive_gym:FeedingJaco-v1', n_envs=n_envs, seed=seed, config=capi.default_config(residual_threshold=0.0))
    env._sim_lib = lib
    return env


def _check_surface(lib):
    env = _make(lib, 1, 1001)
    assert env.action_space.shape == (7,) and env.observation_space.shape == (25,)   # feeding.py:10: 18 + 7
    obs = env.reset()
    assert obs.shape == (25,) and np.all(np.isfinite(obs))
    o, r, d, info = env.step(env.action_space.sample())
    assert o.shape == (25,) and isinstance(r, float) and isinstance(d, bool)
    assert set(info) >= {'total_force_on_human', 'task_success', 'action_robot_len', 'obs_robot_len'}
    # Agent surface
    q = env.robot.get_joint_angles(env.robot.controllable_joint_indices)
    assert q.shape == (7,)
    pos, orient = env.robot.get_pos_orient(env.robot.right_end_effector)
    assert pos.shape == (3,) and orient.shape == (4,) and abs(np.linalg.norm(orient) - 1) < 1e-5
    la, lb, pa, pb, f = env.tool.get_contact_points()
    assert len(la) == len(f)
    assert env.robot.lower_limits[2] == pytest.approx(0.820304748437)               # j2s7s300_joint_2 lower limit
    # done after 200 steps (feeding.py:37)
    for _ in range(199):
        o, r, d, info = env.step(np.zeros(7, dtype=np.float32))
    assert d is True
    env.close()


def _check_fused_vs_api(lib, n_envs, impairment='random'):
    a, b = _make(lib, n_envs, 7), _make(lib, n_envs, 7)
    a.human_impairment = b.human_impairment = impairment
    oa, ob = a.reset(), b.reset()
    if impairment == 'tremor':
        assert len(b.agents) >= 2                     # env.py:130-131: a tremor human is an agent
        # the API path clamps through Human.enforce_joint_limits (agent.py:240-250), the fused path
        # through the integrator's hard-limit flag: switch the flag off on the API side
        for h in b.humans.values():
            b.id.set_hard_limits([h._gl(j) for j in h.controllable_joint_indices], False)
    assert np.allclose(oa, ob, atol=1e-6)
    rng = np.random.default_rng(0)
    for k in range(4):
        act = rng.uniform(-1, 1, size=(n_envs, 7)).astype(np.float32)
        o1, r1, d1, _ = a.step(act if n_envs > 1 else act[0])
        o2, r2, d2, _ = b.step_reference_api(act)
        assert np.abs(np.asarray(o1) - np.asarray(o2)).max() < 1e-4, (k, np.abs(np.asarray(o1) - np.asarray(o2)).max())
        assert np.abs(np.asarray(r1) - np.asarray(r2)).max() < 1e-4
    a.close()
    b.close()


def test_surface_cpu_harness(emu_lib):
    _check_surface(emu_lib)


@pytest.mark.parametrize('impairment', ['random', 'tremor'])
def test_fused_step_equals_reference_api_cpu_harness(emu_lib, impairment):
    _check_fused_vs_api(emu_lib, 2, impairment)


@pytest.mark.gpu
def test_surface_gpu(gpu_lib):
    _check_surface(None)


@pytest.mark.gpu
@pytest.mark.parametrize('impairment', ['random', 'tremor'])
def test_fused_step_equals_reference_api_gpu(gpu_lib, impairment):
    _check_fused_vs_api(None, 8, impairment)


def test_agent_surface_extras(emu_lib):
    """The rest of the reference's Agent surface (agent.py:94-98,132-207,252-283): per-body gravity, AABB heights, IK,
    URDF effort limits; calls that would change the immutable scene template say so."""
    import pytest
    from assistive_gym_b200 import envs
    env = envs.make('FeedingJaco-v1', n_envs=2)
    env._sim_lib = emu_lib
    env.reset()
    sim, robot = env.id, env.robot
    assert all(f > 0 for f in robot.get_joint_max_force(robot.controllable_joint_indices))
    # heights from the link AABBs (agent.py:132-143) against the scene's collider vertices
    height, base_height = env.tool.get_heights()
    assert height.shape == (2,) and np.all(height > 0.005) and np.all(height < 0.3)
    mn, mx = sim.get_link_aabb([int(sim.scene['body_link0'][env.tool.body])])
    assert np.all(mn[:, 0] < mx[:, 0])
    # IK to the current end-effector pose returns a configuration that reproduces it
    ee = robot.right_end_effector
    pos, orient = (np.atleast_2d(a) for a in robot.get_pos_orient(ee))
    q = np.atleast_2d(robot.ik(ee, pos, orient, robot.controllable_joint_indices, max_iterations=200))
    robot.set_joint_angles(robot.controllable_joint_indices, q)
    pos2 = np.atleast_2d(robot.get_pos_orient(ee)[0])
    assert np.abs(pos2 - pos).max() < 0.03
    # per-body gravity (agent.py:196-197): the spoon is released from the arm's pull only through its own gravity
    v0 = np.atleast_2d(env.bowl.get_velocity(env.bowl.base)) if hasattr(env, 'bowl') else None
    env.tool.set_gravity(0, 0, -9.81)
    env.tool.set_gravity(0, 0, 0)
    with pytest.raises(NotImplementedError):
        robot.set_mass(1, 2.0)
    with pytest.raises(NotImplementedError):
        robot.create_constraint(1, env.tool, -1)
    env.close()


def test_cooptimisation_env_dict_interface(emu_lib):
    """FeedingJacoHuman-v1 (reference feeding_envs.py:56-59, feeding.py:13-14,40-43,101-111): dict actions in, dict observations /
    rewards / dones out; the person's head joints follow the human action and respect their limits."""
    from assistive_gym_b200 import envs
    env = envs.make('FeedingJacoHuman-v1', n_envs=2)
    env._sim_lib = emu_lib
    obs = env.reset()
    assert set(obs) == {'robot', 'human'} and obs['robot'].shape == (2, 25) and obs['human'].shape == (2, 23)
    assert env.action_space.shape == (11,) and env.action_robot_len == 7 and env.action_human_len == 4
    active = [env.humans['male' if m else 'female'] for m in env.male]
    q0 = np.stack([np.atleast_2d(h.get_joint_angles(env.human.controllable_joint_indices))[e] for e, h in enumerate(active)])
    rng = np.random.default_rng(0)
    for _ in range(4):
        o, r, d, info = env.step({'robot': rng.uniform(-1, 1, size=(2, 7)), 'human': np.full((2, 4), 1.0)})
    q1 = np.stack([np.atleast_2d(h.get_joint_angles(env.human.controllable_joint_indices))[e] for e, h in enumerate(active)])
    assert np.all(q1 - q0 > 0.01)                                           # a positive action turns every head joint
    lo = np.array([active[0].lower_limits[j] for j in env.human.controllable_joint_indices])
    hi = np.array([active[0].upper_limits[j] for j in env.human.controllable_joint_indices])
    assert np.all(q1 >= lo - 1e-6) and np.all(q1 <= hi + 1e-6)
    assert set(r) == {'robot', 'human'} and np.array_equal(r['robot'], r['human']) and set(d) == {'robot', 'human', '__all__'}
    assert o['human'].shape == (2, 23) and np.all(np.isfinite(o['human'])) and np.allclose(o['human'][:, 10:14], q1, atol=1e-6)
    # the robot part is what the single-agent env reports
    assert np.allclose(o['robot'], env._get_obs('robot'))
    assert info['robot']['action_human_len'] == 4 and info['robot']['obs_human_len'] == 23
    env.close()


def test_realistic_joint_limit_classifier():
    """The joint-limit MLP (reference envs/env.py:39, agents/human.py:134-152) compiled out of the Keras file: layer shapes, and the
    poses the tasks start the person in are reachable while a hyper-extended elbow / a shoulder turned far back are not."""
    from assistive_gym_b200.limits_model import load_model
    m = load_model()
    assert [w.shape for w, _, _ in m.layers] == [(4, 64), (64, 64), (64, 64), (64, 1)] and [a for _, _, a in m.layers] == ['tanh'] * 3 + ['sigmoid']

    def conv(tz, tx, ty, qe, right=True):                       # human.py:141-146
        s = -1 if right else 1
        return [(s * tz + 2 * np.pi) % (2 * np.pi), (tx + 2 * np.pi) % (2 * np.pi), s * ty, (-qe + 2 * np.pi) % (2 * np.pi)]
    d = np.deg2rad
    ok = m.predict_classes([conv(0, 0, 0, 0), conv(d(30), 0, 0, d(-90)), conv(0, 0, 0, d(-90), right=False)])[:, 0]
    bad = m.predict_classes([conv(0, 0, 0, d(90)), conv(d(-150), 0, 0, 0), conv(0, 0, 0, d(-150))])[:, 0]
    assert ok.tolist() == [1, 1, 1] and bad.tolist() == [0, 0, 0]
    p = m.predict(np.random.default_rng(0).uniform(-7, 7, size=(256, 4)))
    assert p.shape == (256, 1) and np.all((p >= 0) & (p <= 1))


def test_keras_file_compiles_to_the_committed_weights():
    """tools/compile_assets.py reads the reference's HDF5 file (an unchanged copy under tests/golden) with its own minimal reader
    (no h5py needed)."""
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref = os.path.join(root, 'tests', 'golden', 'realistic_arm_limits_model.h5')
    sys.path.insert(0, os.path.join(root, 'tools'))
    from compile_assets import compile_keras_mlp
    from assistive_gym_b200.limits_model import load_model
    z = compile_keras_mlp(ref)
    for k, (w, b, act) in enumerate(load_model().layers):
        assert np.array_equal(z['W%d' % k], w) and np.array_equal(z['b%d' % k], b) and str(z['act%d' % k]) == act


def test_cooptimisation_scratch_itch_keeps_the_arm_within_realistic_limits(emu_lib):
    """ScratchItchJacoHuman-v1 (reference scratch_itch_envs.py, scratch_itch.py:11-12,39-44,75-84, env.py:229-231): dict interface; the
    person's right arm follows the human action.  Raising the upper arm sideways: the joint itself goes to 198 degrees, the
    classifier calls everything beyond ~115 degrees (elbow bent) unreachable and sends the arm back to the last reachable pose
    after every substep -- with the check switched off the same actions take the arm past that."""
    from assistive_gym_b200 import envs
    from assistive_gym_b200.limits_model import load_model
    model = load_model()

    def reachable(q):
        tz, tx, ty, qe = q[:, 3], q[:, 4], q[:, 5], q[:, 6]
        x = np.stack([(-tz + 2 * np.pi) % (2 * np.pi), (tx + 2 * np.pi) % (2 * np.pi), -ty, (-qe + 2 * np.pi) % (2 * np.pi)], axis=1)
        return model.predict_classes(x)[:, 0]

    def run(check):
        env = envs.make('ScratchItchJacoHuman-v1', n_envs=2, seed=7)
        env._sim_lib = emu_lib
        orig = env._sb.sample

        def sample(n, rng):                                                  # no impairment: full joint limits, full strength
            smp = orig(n, rng)
            smp['impairment'][:] = 0; smp['limit_scale'] = np.ones(n); smp['strength'] = np.ones(n)
            return smp
        env._sb.sample = sample
        obs = env.reset()
        assert set(obs) == {'robot', 'human'} and obs['robot'].shape == (2, 30) and obs['human'].shape == (2, 34)
        assert env.action_space.shape == (17,) and env.action_robot_len == 7 and env.action_human_len == 10
        active = [env.humans['male' if m else 'female'] for m in env.male]
        ci = env.human.controllable_joint_indices
        if not check:
            for h in env.humans.values():
                h.enforce_realistic_joint_limits = lambda *a, **k: None
        a_h = np.zeros((2, 10)); a_h[:, 3] = 1.0                             # j_right_shoulder_x up
        ok, out = [], None
        for _ in range(45):
            out = env.step({'robot': np.zeros((2, 7)), 'human': a_h})
            q = np.stack([np.atleast_2d(h.get_joint_angles(ci))[e] for e, h in enumerate(active)])
            ok.append(reachable(q))
        env_obs_robot = env._get_obs('robot')
        env.close()
        return q, np.array(ok), out, env_obs_robot
    q_on, ok_on, (o, r, d, info), robot_obs = run(True)
    q_off, ok_off, _, _ = run(False)
    assert np.all(ok_on == 1)                                               # every step ended in a reachable pose
    assert np.all(q_on[:, 3] > np.deg2rad(60)) and np.all(q_on[:, 3] < np.deg2rad(125))
    assert np.all(q_off[:, 3] > np.deg2rad(135)) and not np.all(ok_off == 1)  # without the check the arm goes on
    assert set(r) == {'robot', 'human'} and np.array_equal(r['robot'], r['human']) and set(d) == {'robot', 'human', '__all__'}
    assert o['human'].shape == (2, 34) and np.all(np.isfinite(o['human'])) and np.allclose(o['human'][:, 13:23], q_on, atol=1e-6)
    assert np.allclose(o['robot'], robot_obs)
    assert info['robot']['action_human_len'] == 10 and info['robot']['obs_human_len'] == 34


def test_limits_impairment_scales_the_controllable_arm_limits(emu_lib):
    """impairment 'limits' (human.py:85, human_creation.py:217-218): in the co-optimisation env the person's joint limits are scaled
    per env; the start pose is clipped to them and the arm cannot be driven past them."""
    from assistive_gym_b200 import envs
    env = envs.make('ScratchItchJacoHuman-v1', n_envs=2, seed=3)
    env._sim_lib = emu_lib
    orig = env._sb.sample

    def sample(n, rng):
        s = orig(n, rng)
        s['impairment'][:] = [1, 0]; s['limit_scale'] = np.array([0.5, 1.0]); s['strength'][:] = 1.0
        return s
    env._sb.sample = sample
    env.reset()
    active = [env.humans['male' if m else 'female'] for m in env.male]
    elbow = lambda: np.array([np.atleast_2d(h.get_joint_angles([6]))[e, 0] for e, h in enumerate(active)])
    q0 = elbow()
    assert abs(q0[0] - np.deg2rad(-64)) < 1e-4 and abs(q0[1] - np.deg2rad(-90)) < 1e-4      # -128 degrees x 0.5; the preset elsewhere
    a_h = np.zeros((2, 10)); a_h[:, 6] = -1.0                                            # bend the elbow further
    for _ in range(12):
        env.step({'robot': np.zeros((2, 7)), 'human': a_h})
    q1 = elbow()
    assert q1[0] >= np.deg2rad(-64) - 1e-5 and q1[1] < np.deg2rad(-95)
    env.close()
