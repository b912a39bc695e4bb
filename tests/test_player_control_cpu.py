"""CPU: argument validation of the player entry point of the dynamics step (tb_dyn_step_player) and the CPU reference
of caller control (tests/_player_oracle.py) against the oracle's rollout."""
import pytest
import torch

from oracle import tb_oracle as O
from trafficbotsv1_5_b200 import config, lib, params, synth

from _player_oracle import dynamics_update, rollout

TB_ERR_BAD_SHAPE, TB_ERR_NULL = -1, -5


@pytest.fixture(scope="module")
def handle():
    lib.build()
    return lib.load()


def _dyn_args(one, B=2, A=3, W=11, T=5, n_gt=6, player_valid=None, player_action=None, **over):
    """tb_dyn_step_player arguments with fake device pointers (never dereferenced: validation fails first)."""
    a = dict(act_branch=one, ag_type=one, max_acc=one, max_yaw_rate=one, dt=0.1, valid=one, disabled=one,
             navi_invalid=one, dest_reached=one, pose=one, motion=one, gt_valid=one, gt_pose=one, gt_motion=one,
             tf_mask=one, n_gt=n_gt, sc_div=1, boundary=one, dest_idx=one, mp_pos=one, mp_dirn=one,
             mp_node_invalid=one, mp_kind=one, n_mp=4, n_node=20, thresh_lane=50.0, thresh_edge=10.0, cos_rot=0.866,
             d_step=one, B=B, A=A, W=W, T=T, hist_valid=one, hist_pose=one, hist_motion=one, pred_valid=one,
             pred_pose=one, pred_motion=one, o_outside=None, o_reached=None, player_valid=player_valid,
             player_action=player_action, stream=None)
    a.update(over)
    return list(a.values())


def test_dyn_step_player_error_codes_without_gpu(handle):
    one = 16  # any non-null, 16-byte aligned fake address
    f = handle.tb_dyn_step_player
    assert f(*_dyn_args(one, player_valid=one, player_action=None)) == TB_ERR_NULL  # a plan is required with players
    assert f(*_dyn_args(one, pose=None, player_valid=one, player_action=one)) == TB_ERR_NULL
    assert f(*_dyn_args(one, d_step=None)) == TB_ERR_NULL
    assert f(*_dyn_args(one, B=0, player_valid=one, player_action=one)) == TB_ERR_BAD_SHAPE
    assert f(*_dyn_args(one, T=0, player_valid=one, player_action=one)) == TB_ERR_BAD_SHAPE
    assert f(*_dyn_args(one, n_gt=0)) == TB_ERR_BAD_SHAPE
    assert f(*_dyn_args(one, sc_div=0, player_valid=one, player_action=one)) == TB_ERR_BAD_SHAPE
    # tb_dyn_step_ex = the same arguments without the two player pointers
    assert handle.tb_dyn_step_ex(*(_dyn_args(one, B=0)[:-3] + [None])) == TB_ERR_BAD_SHAPE
    assert handle.tb_dyn_step_ex(*(_dyn_args(one, valid=None)[:-3] + [None])) == TB_ERR_NULL


def test_dynamics_update_player_override():
    """The override replaces the physical action of valid player agents only; invalid or untyped agents stay zero."""
    g = torch.Generator().manual_seed(0)
    B, A = 2, 6
    pose, motion, mean = torch.randn(B, A, 3, generator=g), torch.randn(B, A, 3, generator=g), torch.randn(B, A, 2, generator=g)
    valid = torch.ones(B, A, dtype=torch.bool)
    valid[0, 1] = False
    ag_type = torch.zeros(B, A, 3, dtype=torch.bool)
    ag_type[:, :, 0] = True
    ag_type[1, 2] = False
    pv = torch.zeros(B, A, dtype=torch.bool)
    pv[:, :3] = True
    pa = torch.randn(B, A, 2, generator=g) * 3
    dyn = config.DYNAMICS_CFG
    p0, m0 = O.dynamics_update(pose, motion, valid, ag_type, mean, dyn)
    p1, m1 = dynamics_update(pose, motion, valid, ag_type, mean, dyn)
    assert torch.equal(p0, p1) and torch.equal(m0, m1)
    p2, m2 = dynamics_update(pose, motion, valid, ag_type, mean, dyn, pv, pa)
    on = pv & valid & ag_type.any(-1)
    assert torch.equal(m2[..., 1:][on], pa[on])
    assert torch.equal(p2[~on], p0[~on]) and torch.equal(m2[~on], m0[~on])
    assert float(p2[0, 1].abs().max()) == 0.0 and float(p2[1, 2].abs().max()) == 0.0


def test_player_oracle_without_control_is_the_oracle():
    cfg = config.default_model_cfg()
    P = params.init_params(cfg, seed=0)
    batch = synth.make_scene_batch(n_sc=1, n_ag=28, n_mp=70, n_tl=27, seed=5, boundary=103.0)
    sz = config.derived_sizes(cfg)
    R, T = 2, 14
    ref = O.rollout(P, cfg, sz, config.DYNAMICS_CFG, config.ROLLOUT_CFG, batch, R, T)
    res = rollout(P, cfg, sz, config.DYNAMICS_CFG, config.ROLLOUT_CFG, batch, R, T)
    for k in ("pred_valid", "pred_pose", "pred_motion", "tl_state", "final_valid", "final_navi_valid"):
        assert torch.equal(res[k], ref[k]), k
