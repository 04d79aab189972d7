"""Host-side logic: task ids, observation indexing, datasets, rewards, has_fallen, TaskSpec packing (CPU only)."""
import os

import numpy as np
import pytest

from helpers import golden, make_env, blobs, ROOT


def test_task_names_and_registry():
    import loco_mujoco_b200 as lm
    names = lm.get_all_task_names()
    assert "UnitreeA1.simple.real" in names and "UnitreeA1.hard.real" in names
    assert "UnitreeA1" in lm.LocoEnv.list_registered_loco_mujoco()
    with pytest.raises(ValueError):
        lm.LocoEnv.make("UnitreeA1.nonexistent")


def test_a1_spaces_and_indexing(bundled_only):
    env = make_env("UnitreeA1.simple")
    assert env.info.observation_space.shape == (37,)
    assert env.info.action_space.shape == (12,)
    assert np.all(env.info.action_space.low == -1) and np.all(env.info.action_space.high == 1)
    assert env.dt == pytest.approx(0.01)
    # index contract of the reference docstring table (unitreeA1.py:50-164)
    assert env.get_obs_idx("q_trunk_tz") == [0]
    assert env.get_obs_idx("q_FR_hip_joint") == [4]
    assert env.get_obs_idx("dq_trunk_tx") == [16]
    lo, hi = env.info.observation_space.low, env.info.observation_space.high
    assert lo[0] == -np.inf and hi[4] == pytest.approx(0.802851) and lo[6] == pytest.approx(-2.69653)
    assert list(lo[-3:]) == [-1, -1, -np.inf]


def test_reset_row_bit_exact_vs_golden(bundled_only):
    """reset = trajectory table lookup + goal features; no physics involved."""
    for task in ("UnitreeA1.simple", "UnitreeA1.hard"):
        env = make_env(task)
        g = golden(task)
        spec = env.task_spec()
        np.random.seed(0)
        np.random.randint(0, 1)
        tr = np.random.randint(0, env.trajectories.number_of_trajectories)
        st = np.random.randint(0, env.trajectories.trajectory_length)
        row = spec.table[tr, st].copy()
        nq = env._model.nq
        row[spec.recenter] = 0
        src = {0: row[:nq], 1: row[nq:2 * nq], 2: row[2 * nq:]}
        obs = np.array([src[t][i] for t, i in zip(spec.obs_src_type, spec.obs_src_idx)])
        assert np.abs(obs - g[0]).max() < 1e-13


def test_create_dataset_and_has_fallen(bundled_only):
    env = make_env("UnitreeA1.simple")
    d = env.create_dataset()
    n_traj, T = env.trajectories.number_of_trajectories, env.trajectories.trajectory_length
    assert d["states"].shape == (n_traj * (T - 1), 37) and d["next_states"].shape == d["states"].shape
    assert d["last"].sum() == n_traj and d["absorbing"].sum() == 0
    assert np.allclose(d["states"][1], d["next_states"][0])
    g = golden("UnitreeA1.simple")
    assert env._has_fallen(g[-1]) and not env._has_fallen(g[0])
    assert env.is_absorbing(g[-1])


def test_rewards_match_definitions():
    from loco_mujoco_b200.utils import VelocityVectorReward, TargetVelocityReward, PosReward, NoReward, CustomReward
    s = np.arange(10, dtype=float) * 0.1
    assert NoReward()(s, None, s, False) == 0
    assert PosReward(3)(s, None, s, False) == pytest.approx(0.3)
    assert TargetVelocityReward(1.25, 4)(s, None, s, False) == pytest.approx(np.exp(-(0.4 - 1.25) ** 2))
    r = VelocityVectorReward(0, 1, [-3, -2], [-1])(s, None, s, False)
    assert r == pytest.approx(np.exp(-5 * np.linalg.norm(np.array([0.0, 0.1]) - 0.9 * np.array([0.7, 0.8]))))
    assert CustomReward(lambda a, b, c: 7.0)(s, None, s, False) == 7.0


def test_taskspec_pack_layout(bundled_only):
    env = make_env("UnitreeA1.simple")
    (mi, mr), (ti, tr) = blobs(env)
    assert ti[0] == 0x5441534B and ti[2] == 37 and ti[5] == 10
    n_traj, T, ncol = env.task_spec().table.shape
    assert ncol == 2 * 18 + 3
    assert len(tr) == 8 + 12 + 12 + 3 + 3 + n_traj * T * ncol
    assert mi[0] == 0x4C4F434F and mi[2] == env._model.nbody and mi[3] == 18


def test_bundled_assets_match_live_compile(bundled_only):
    """The bundled UnitreeA1.simple asset packs to exactly the ModelPack / TaskSpec blobs that a live compile of a
    loco-mujoco checkout gives (MJCF + mini dataset; LOCO_MUJOCO_PATH set, bundled assets not forced), stored in
    tests/golden/UnitreeA1.simple.live_compile.npz as a0, a1 (modelpack.pack) and t0, t1 (TaskSpec.pack)."""
    from loco_mujoco_b200 import modelpack
    e = make_env("UnitreeA1.simple")
    a, t = modelpack.pack(e._model), e.task_spec().pack()
    live = np.load(os.path.join(ROOT, "tests", "golden", "UnitreeA1.simple.live_compile.npz"))
    for k, x in zip(("a0", "a1", "t0", "t1"), (*a, *t)):
        assert np.array_equal(live[k], x), k


def test_taskspec_layout_and_feature_sources(bundled_only):
    """Wire format of the task description (include/locosim_task.h, version 4): header fields and array lengths."""
    from loco_mujoco_b200 import task as T
    env = make_env("UnitreeA1.simple", use_foot_forces=True)
    spec = env.task_spec()
    ints, reals = spec.pack()
    assert ints[0] == T.MAGIC and ints[1] == T.VERSION == 4 and ints[2] == spec.obs_dim == 49
    assert ints[16] == 4 and ints[17] == env._model.ngeom                      # TKI_N_GRF, TKI_N_GRF_GEOM
    nu = len(spec.act_idx)
    assert list(ints[18:21]) == [-1, -1, -1]                                      # TKI_ROT_*: setup_random_rot off
    assert len(ints) == 24 + 2 * spec.obs_dim + len(spec.done_terms) + nu + env._model.ngeom
    n_traj, T_len, ncol = spec.table.shape
    assert len(reals) == 8 + 2 * nu + 2 * len(spec.done_terms) + n_traj * T_len * ncol
    assert list(spec.obs_src_type[-12:]) == [T.OBS_GRF] * 12 and list(spec.obs_src_idx[-12:]) == list(range(12))
    groups = spec.grf_group
    assert (groups == T.GRF_FLOOR).sum() == 1 and sorted(groups[groups >= 0][groups[groups >= 0] < 127].tolist()) == [0, 1, 2, 3]


def test_multi_model_envs_are_parameter_pools(bundled_only):
    """Carry tasks: one model per weight, pooled; the weight is a user feature of the pool row (OBS_PARAM)."""
    from loco_mujoco_b200 import task as T
    from loco_mujoco_b200.domain_randomization import POOL_FIELDS, N_USER
    env = make_env("Atlas.carry")
    assert len(env._models) == 4 and [u[0] for u in env._model_user_features] == [0.1, 1.0, 5.0, 10.0]
    spec = env.task_spec()
    assert spec.obs_src_type[-1] == T.OBS_PARAM and spec.obs_src_idx[-1] == 0
    assert env.info.observation_space.shape == (31,) and env.info.observation_space.low[-1] == 0.1
    pool = env.model_pool()
    m = env._model
    dims = dict(nv=m.nq, nbody=m.nbody, ngeom=m.ngeom)
    n = sum(dims[k] * c for _, k, c in POOL_FIELDS) + 1 + N_USER
    assert pool.shape == (4, n + (-n) % 4)
    assert np.allclose(pool[:, n - N_USER], [0.1, 1.0, 5.0, 10.0]) and not np.allclose(pool[0], pool[3])
    # the heavier box shows up in the torso's mass only
    mass = np.array([mm.body_mass for mm in env._models])
    assert np.count_nonzero(np.abs(mass[3] - mass[0]) > 1e-9) == 1 and abs((mass[3] - mass[0]).sum() - 9.9) < 1e-9


def test_humanoid_4ages_modes(bundled_only):
    env = make_env("HumanoidTorque4Ages.run.2")
    assert env._model_user_features == [(0.0, 1.0)] and env.info.observation_space.shape == (38,)
    assert abs(env._reward_params["target_velocity"] - 2.5 * 0.6) < 1e-12      # MultiTargetVelocityReward: target x scaling
    # mode "all": a composite of the four single-scaling envs (one engine each, created lazily)
    env = make_env("HumanoidTorque4Ages.run.all")
    assert type(env).__name__ == "HumanoidTorque4AgesAll" and len(env.subs) == 4 and not env.batched
    assert env.info.observation_space.shape == (38,) and env.info.action_space.shape == (13,)
    assert [s._model_user_features[0] for s in env.subs] == [(0.0, 0.0), (0.0, 1.0), (1.0, 0.0), (1.0, 1.0)]
    assert sum(len(s.create_dataset()["states"]) for s in env.subs) == len(env.create_dataset()["states"])
    with pytest.raises(ValueError):
        make_env("HumanoidTorque4Ages.run.all", num_envs=3)


def test_vector_wrapper_spaces(bundled_only):
    from loco_mujoco_b200 import VectorGymnasiumWrapper
    v = VectorGymnasiumWrapper("UnitreeG1.run.real", num_envs=8, debug=True)       # no engine until reset()
    assert v.observation_space.shape == (8, 56) and v.action_space.shape == (8, 23)
    assert v.single_observation_space.shape == (56,) and v.metadata["autoreset_mode"] == "same_step"


def test_get_mask_pomdp(bundled_only):
    """POMDP masks (base_robot_humanoid.py:38-90): parts of the observation by name, in observation order."""
    e = make_env("Atlas.carry")
    m = e.get_mask(("velocities", "weight"))
    assert m.shape == (31,) and m[:14].all() and not m[14:].any()
    e = make_env("Talos.walk", use_foot_forces=True)
    m = e.get_mask("foot_forces")
    assert m.shape == e.info.observation_space.shape == (40,) and m[:34].all() and not m[34:].any()
    with pytest.raises(AssertionError):
        make_env("Talos.walk").get_mask("foot_forces")


def test_unitree_h1_carry_builds(bundled_only):
    """UnitreeH1.carry (unitreeH1.py:235-296,425-444): four weight models, the weight is observed. No golden row beyond
    the reset row pins it (H1's mesh-foot contacts, DESIGN.md section 7), so there is no parity test for it."""
    env = make_env("UnitreeH1.carry")
    assert len(env._models) == 4 and env.info.observation_space.shape == (33,)
    assert [u[0] for u in env._model_user_features] == [0.1, 1.0, 5.0, 10.0]


def test_tracking_reward_spec_on_the_oracle(oracle, bundled_only):
    """reward_type="tracking" (include/locosim_task.h LS_REWARD_TRACKING): the oracle's reward equals the formula evaluated
    in numpy on its own post-step observation and the table row at the advanced cursor; TaskSpec v4 carries the weights."""
    from helpers import make_env, blobs
    env = make_env("HumanoidTorque.run", reward_type="tracking", reward_params=dict(k_pose=1.5))
    spec = env.task_spec()
    assert spec.reward_type == 4 and spec.tracking == [0.7, 1.5, 0.3, 0.1] and spec.random_rot == [-1, -1, -1]
    ints, reals = spec.pack()
    assert ints[1] == 4 and list(reals[2:6]) == spec.tracking
    oe = oracle.env(*blobs(env))
    oe.reset_to(0, 10)
    nq = env._model.nq
    rng = np.random.RandomState(0)
    for k in range(5):
        obs, r, done = oe.step(rng.uniform(-1, 1, env._model.nu))
        row = spec.table[0, min(10 + k + 1, spec.table.shape[1] - 1)]
        ep = sum((obs[j] - row[i]) ** 2 for j, (t, i) in enumerate(zip(spec.obs_src_type, spec.obs_src_idx)) if t == 0)
        ev = sum((obs[j] - row[nq + i]) ** 2 for j, (t, i) in enumerate(zip(spec.obs_src_type, spec.obs_src_idx)) if t == 1)
        assert abs(r - (0.7 * np.exp(-1.5 * ep) + 0.3 * np.exp(-0.1 * ev))) < 1e-12
    oe.close()


def test_random_rotation_spec(bundled_only):
    from helpers import make_env
    env = make_env("UnitreeA1.simple", setup_random_rot=True)
    m = env._model
    assert env.task_spec().random_rot == [m.joint_id("trunk_rotation"), m.joint_id("trunk_tx"), m.joint_id("trunk_ty")]
    assert make_env("UnitreeA1.simple").task_spec().random_rot == [-1, -1, -1]
