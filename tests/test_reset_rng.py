"""Reset randomisation, draw for draw (SURVEY.md 8-a11).

The reference draws every reset from numpy's RandomState(config.seed) (furniture.py:72; seed + rank per VecEnv worker,
env/base.py:77): the placement sampler (placement_sampler.py:137-190) and 101 robot-noise vectors (furniture.py:1581, :1609).
tests/golden/placement.npz holds what the reference's OWN sampler code produces (tools/make_golden_placement.py).  Checked:
  * the oracle's restatement of the sampler against those vectors: bit-exact;
  * the device generator (MT19937 state per env in HBM, numpy's double and uniform formulas) against numpy itself: the
    state after three resets is bit-identical, so every draw was;
  * the device reset against the oracle env seeded the same way: same placements, same settled state to fp32 round-off."""
import os

import numpy as np
import pytest

from furniture_b200 import mjcf
from oracle.ref_env import Cfg, OracleFurnitureEnv
from parity_util import make_engine

BACKENDS = [pytest.param(False, id="emu"), pytest.param(True, id="cuda", marks=pytest.mark.gpu)]
G = np.load(os.path.join(os.path.dirname(__file__), "golden", "placement.npz"))
FURN = ["table_lack_0825", "swivel_chair_0700"]


@pytest.mark.parametrize("furn", FURN)
def test_oracle_placement_is_the_reference_sampler(furn):
    m = mjcf.load_scene("Sawyer", furn)
    for si, seed in enumerate(G[furn + "/seeds"]):
        cfg = Cfg()
        cfg.seed = int(seed)
        e = OracleFurnitureEnv(m, cfg)
        for r in range(G[furn + "/pos"].shape[1]):
            pl = e.place()
            assert np.array_equal(np.array([p for p, _ in pl]), G[furn + "/pos"][si, r])
            assert np.array_equal(np.array([q for _, q in pl]), G[furn + "/quat"][si, r])
            for _ in range(101):
                nz = e.rng.uniform(-cfg.agent_xyz_rand, cfg.agent_xyz_rand, e.narm)
            assert np.array_equal(nz, G[furn + "/noise"][si, r])
        st = e.rng.get_state()
        assert np.array_equal(st[1], G[furn + "/mt"][si]) and st[2] == G[furn + "/mtpos"][si]


@pytest.mark.parametrize("gpu", BACKENDS)
@pytest.mark.parametrize("furn", FURN)
def test_device_generator_is_numpy_randomstate(furn, gpu):
    """env i of a handle seeded s owns RandomState(s + i); golden seeds 123 and 124 are two consecutive envs"""
    m = mjcf.load_scene("Sawyer", furn)
    eng = make_engine(m, 2, gpu, seed=123)
    nreset = G[furn + "/pos"].shape[1]
    for r in range(nreset):
        eng.env_reset()
    st, pos = eng.get("mt_state"), eng.get("mt_pos")[:, 0]
    for i in range(2):
        assert pos[i] == G[furn + "/mtpos"][i]
        assert np.array_equal(st[i], G[furn + "/mt"][i])
    assert (eng.get("flags") == 0).all()
    eng.close()


@pytest.mark.parametrize("gpu", BACKENDS)
@pytest.mark.parametrize("furn", FURN)
def test_reset_equals_the_oracle_env_seeded_the_same_way(furn, gpu):
    m = mjcf.load_scene("Sawyer", furn)
    n, seed = 3, 500
    eng = make_engine(m, n, gpu, seed=seed)
    envs = []
    for i in range(n):
        cfg = Cfg()
        cfg.seed = seed + i
        envs.append(OracleFurnitureEnv(m, cfg))
    for r in range(2):  # the second reset continues the stream
        eng.env_reset()
        q, v = eng.get("qpos"), eng.get("qvel")
        for i, e in enumerate(envs):
            e.reset()
            # 300 mj_steps of settling in fp32 vs fp64 from identical placements (cylinder contacts go through MPR, whose
            # portal tolerance bounds depth to ~1e-5: looser for the chair)
            tol = 1e-5 if furn == "table_lack_0825" else 1e-4
            assert np.abs(q[i] - e.sim.qpos).max() < tol, (r, i, np.abs(q[i] - e.sim.qpos).max())
            assert np.abs(v[i] - e.sim.qvel).max() < 2e-4
    assert np.abs(q[0, 9:11] - q[1, 9:11]).max() > 1e-4  # different envs, different placements
    eng.close()


def test_masked_reset_touches_only_the_selected_envs():
    """fe_env_reset(mask): the envs whose mask byte is set are reset (their random stream continues: second reset of the
    oracle env seeded the same way), the others keep state, bookkeeping and generator untouched (lane-emulated build: the
    mask pointer is a host pointer there, a device pointer for the CUDA library)."""
    m = mjcf.load_scene("Sawyer", "table_lack_0825")
    n, seed = 3, 900
    eng = make_engine(m, n, False, seed=seed, nsub=5)
    eng.env_reset()
    a = np.random.RandomState(1).uniform(-1, 1, (n, eng.act_dim)).astype(np.float32)
    a[:, -1] = -1
    eng.env_step_host(a)
    q1, mt1, len1 = eng.get("qpos").copy(), eng.get("mt_state").copy(), eng.get("episode_length").copy()
    mask = np.array([1, 0, 1], dtype=np.uint8)
    eng.env_reset(mask_dev=mask.ctypes.data)
    q2, len2 = eng.get("qpos"), eng.get("episode_length")
    assert np.array_equal(q2[1], q1[1]) and np.array_equal(eng.get("mt_state")[1], mt1[1]) and len2[1, 0] == len1[1, 0] == 1
    assert len2[0, 0] == 0 and len2[2, 0] == 0
    for i in (0, 2):
        cfg = Cfg()
        cfg.seed = seed + i
        e = OracleFurnitureEnv(m, cfg)
        e.reset()
        e.reset()
        assert np.abs(q2[i] - e.sim.qpos).max() < 1e-5, i


def test_unstable_episode_resets_twice_like_the_reference_worker():
    """MujocoException path (furniture.py:2889-2897): the env resets inside the step, _after_step counts the step and ends the
    episode with the unstable penalty, and the VecEnv worker resets once more (subproc_vec_env.py:16-20).  So after the step
    the episode length is 0 and the env's generator has consumed two more resets' worth of draws; the next step is step 1 of a
    fresh episode.  The divergence guard (|qvel| > 1e6, mj_checkVel) is tripped by planting a huge velocity."""
    m = mjcf.load_scene("Sawyer", "table_lack_0825")
    n, seed = 2, 321
    eng = make_engine(m, n, False, seed=seed, nsub=2)
    eng.env_reset()
    v = eng.get("qvel").copy()
    v[1, 0] = 1e8
    eng.set("qvel", v)
    a = np.zeros((n, eng.act_dim), np.float32)
    a[:, -1] = -1
    obs, rew, done, info = eng.env_step_host(a)
    assert not done[0] and done[1] and info[1][2] == 1 and info[0][2] == 0
    assert rew[1] < -50  # unstable_penalty_coef = 100 (config/furniture.py)
    ln, pos, st = eng.get("episode_length")[:, 0], eng.get("mt_pos")[:, 0], eng.get("mt_state")
    assert ln[0] == 1 and ln[1] == 0
    for i, nreset in ((0, 1), (1, 3)):
        cfg = Cfg()
        cfg.seed = seed + i
        e = OracleFurnitureEnv(m, cfg)
        for _ in range(nreset):
            e.place()
            for _ in range(101):
                e.rng.uniform(-cfg.agent_xyz_rand, cfg.agent_xyz_rand, e.narm)
        s = e.rng.get_state()
        assert s[2] == pos[i] and np.array_equal(s[1], st[i]), i
    assert np.isfinite(obs).all() and (eng.get("flags")[:, 0] & 8 == 0).all()
    obs, rew, done, info = eng.env_step_host(a)
    assert info[1][3] == 1 and info[0][3] == 2 and not done.any()


def test_furn_size_rand_scales_the_scene_and_keeps_the_draw_order():
    """furn_size_rand (config/furniture.py:196-201): the size factor is the first draw of the env's generator (furniture.py:1989-1991)
    and every reset spends one more (:1428-1431); xml_adjusting/rescale.py scales geoms, sites and body offsets of the parts"""
    r, seed = 0.1, 77
    factor = 1 + np.random.RandomState(seed).uniform(-r, r, 1)[0]
    m0 = mjcf.load_scene("Sawyer", "table_lack_0825")
    if mjcf.default_assets_root() is not None:
        m = mjcf.load_scene("Sawyer", "table_lack_0825", resize_factor=factor)
    else:  # a resized scene is composed from the asset tree: without one, the scene it gave (tools/make_golden_resized.py)
        m = mjcf.Model.load(os.path.join(os.path.dirname(__file__), "golden", "table_lack_resized.npz"))
        assert m.meta["resize_factor"] == factor
    g0 = m0.names["geom"].index("noviz_collision_4_part4_0") if "noviz_collision_4_part4_0" in m0.names["geom"] else [i for i, n in enumerate(m0.names["geom"]) if "part4" in n][0]
    assert np.allclose(m.geom_size[g0], m0.geom_size[g0] * factor) and np.allclose(m.geom_pos[g0], m0.geom_pos[g0] * factor)
    s = [i for i, n in enumerate(m0.names["site"]) if "conn_site" in n][0]
    assert np.allclose(m.site_pos[s], m0.site_pos[s] * factor)
    assert np.allclose(m.meta["part_init_qpos"]["4_part4"], m0.meta["part_init_qpos"]["4_part4"])  # *_initpos numerics are not rescaled
    assert np.array_equal(m.geom_size[m.names["geom"].index("FLOOR")], m0.geom_size[m0.names["geom"].index("FLOOR")])
    n = 2
    eng = make_engine(m, n, False, seed=seed, furn_size_rand=r)
    envs = []
    for i in range(n):
        cfg = Cfg()
        cfg.seed, cfg.furn_size_rand = seed + i, r
        envs.append(OracleFurnitureEnv(m, cfg))
    assert abs(envs[0].resize_factor - factor) < 1e-15
    for k in range(2):
        eng.env_reset()
        for i, e in enumerate(envs):
            e.reset()
            st = e.rng.get_state()
            assert eng.get("mt_pos")[i, 0] == st[2] and np.array_equal(eng.get("mt_state")[i], st[1]), (k, i)
            assert np.abs(eng.get("qpos")[i] - e.sim.qpos).max() < 1e-5
    eng.close()
