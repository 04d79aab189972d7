"""Domain randomisation: host semantics (CPU) and pooled per-env parameters on the GPU vs the oracle."""
import copy
import os

import numpy as np
import pytest

from helpers import GOLDEN, make_env, oracle_step_sensitivity

# loco-mujoco's Atlas MJCF (environments/data/atlas/atlas.xml), verbatim; its meshes are visual only, so it compiles alone
ATLAS_XML = os.path.join(GOLDEN, "atlas.xml")

CONF = {"Default": {"exclude": ["pelvis_tx", "pelvis_tz", "pelvis_ty", "pelvis_tilt", "pelvis_list", "pelvis_rotation"],
                    "Joints": {"damping": {"sigma": 0.0}}},
        "Joints": {"hip_flexion_r": {"damping": {"uniform_range": [1.0, 3.0]}, "armature": {"sigma": 0.002}},
                   "knee_angle_l": {"damping": {"sigma": 0.1}, "frictionloss": {"sigma": 0.05}}},
        "Inertial": {"l_uleg": {"mass": {"sigma": 0.5}}, "r_foot": {"diaginertia": {"uniform_range_delta": 0.0005}}}}


def test_apply_domain_randomization_semantics():
    from loco_mujoco_b200 import mjcf
    from loco_mujoco_b200.domain_randomization import apply_domain_randomization, pool_row
    h = mjcf.XmlHandle(ATLAS_XML)
    np.random.seed(0)
    conf = copy.deepcopy(CONF)
    apply_domain_randomization(h, conf)
    j = h.find("joint", "hip_flexion_r")
    assert 1.0 <= float(j.get("damping")) <= 3.0 and float(j.get("armature")) >= 0.0
    # a joint only covered by Default gets an explicit element-level damping centred on 0.0 (class defaults invisible)
    assert float(h.find("joint", "ankle_angle_r").get("damping")) == 0.0
    assert h.find("joint", "pelvis_tx").get("damping") == "0"          # excluded: untouched
    m0 = float(h.find("body", "l_uleg").find("inertial").get("mass"))
    apply_domain_randomization(h, conf)                                  # second call compounds on the mutated handle
    m1 = float(h.find("body", "l_uleg").find("inertial").get("mass"))
    assert m0 != m1
    model = mjcf.compile_model(h, timestep=0.001)
    row = pool_row(model)
    assert len(row) % 4 == 0 and np.isfinite(row).all()
    with pytest.raises(AssertionError):                                  # fullinertia DR needs a fullinertia attribute
        apply_domain_randomization(h, {"Inertial": {"l_uleg": {"fullinertia": {"uniform_range_delta": 0.001}}}})


@pytest.mark.gpu
def test_pooled_parameters_match_oracle(oracle, bundled_only):
    """Fixture tests/golden/dr_atlas_pool.npz = 6 seeded randomised recompilations (tools/make_dr_fixture.py)."""
    torch = pytest.importorskip("torch")
    from helpers import GOLDEN
    fx = np.load(os.path.join(GOLDEN, "dr_atlas_pool.npz"))
    pool, mints, mreals = fx["pool"], fx["model_ints"], fx["model_reals"]
    n = 48
    env = make_env("Atlas.walk", num_envs=n, seed=4)
    eng = env._get_engine()
    assert np.abs(pool - pool[0]).max() > 1e-3
    eng.set_param_pool(pool)
    rng = np.random.RandomState(0)
    tr = np.zeros(n, dtype=np.int32)
    st = rng.randint(0, env.trajectories.trajectory_length, n).astype(np.int32)
    eng.reset(traj_no=torch.tensor(tr, device=eng.device), step_no=torch.tensor(st, device=eng.device))
    rows = eng.param_rows().cpu().numpy()
    assert len(set(rows.tolist())) > 1, "every env drew the same pool row"
    tb = env.task_spec().pack()
    oes = [oracle.env((mints, mreals[r]), tb) for r in rows]
    base = [oracle.env((mints, mreals[(r + 1) % len(pool)]), tb) for r in rows]     # deliberately the WRONG row
    for i in range(n):
        oes[i].reset_to(tr[i], st[i])
        base[i].reset_to(tr[i], st[i])
    wrong_gap, alive, n_switch = 0.0, np.ones(n, dtype=bool), 0
    for k in range(2):
        act = rng.uniform(-1, 1, (n, eng.action_dim)).astype(np.float32)
        obs, rew, done, _ = eng.step(torch.tensor(act, device=eng.device), auto_reset=False)
        obs = obs.cpu().numpy()
        for i in range(n):
            if not alive[i]:
                continue
            q, v = oes[i].get_state()
            o, r, d = oes[i].step(act[i].astype(np.float64))
            ow, _, _ = base[i].step(act[i].astype(np.float64))
            if not np.allclose(obs[i], o, rtol=3e-3 * (k + 1), atol=3e-3 * (k + 1)):
                # only acceptable on a contact / joint-limit switch, where the fp64 result itself jumps as much
                err = np.abs(obs[i] - o).max()
                gap = oracle_step_sensitivity(oracle, (mints, mreals[rows[i]]), tb, tr[i], st[i], q, v, act[i], o)
                assert err < 2.0 * gap, (k, i, err, gap)
                n_switch += 1
                alive[i] = False
                continue
            wrong_gap = max(wrong_gap, np.abs(obs[i] - ow).max())
    assert n_switch <= n // 16, "too many envs disagree with the oracle: %d" % n_switch
    assert wrong_gap > 0.05, "the randomised parameters do not influence the dynamics?"
