"""CPU: argument validation of tb_rule_check and the scenes of tests/_rule_scenes.py (the fp32 and float64 oracles
agree on them, every hand-placed case has the flag pattern it was built for, and the crowd / dense-map scenes overflow
the kernel's candidate queues)."""
import pytest
import torch

import _rule_scenes as RS
from trafficbotsv1_5_b200 import lib

TB_ERR_BAD_SHAPE, TB_ERR_UNSUPPORTED, TB_ERR_NULL = -1, -3, -5
PTRS = ("pred_valid", "pred_pose", "pred_motion", "ag_type", "ag_size", "hist_tl", "tl_invalid", "tl_pose", "seg",
        "node_invalid", "poly_circle", "poly_kind", "passive_counter", "o_collided", "o_collided_wosac",
        "o_run_road_edge", "o_run_red_light", "o_passive", "d_step")
DIMS = ("n_mp", "n_node", "B", "A", "T", "W", "n_tl", "sc_div", "tl_div")


@pytest.fixture(scope="module")
def handle():
    lib.build()
    return lib.load()


def _args(one, **over):
    """tb_rule_check arguments with fake device pointers (never dereferenced: validation fails first)."""
    a = {k: one for k in PTRS}
    a.update(n_mp=8, n_node=20, B=6, A=32, T=10, W=11, n_tl=4, sc_div=3, tl_div=3)
    a.update(over)
    return [a[k] for k in PTRS[:12]] + [a["n_mp"], a["n_node"]] + [a[k] for k in PTRS[12:]] + \
        [a[k] for k in ("B", "A", "T", "W", "n_tl", "sc_div", "tl_div")] + [1.1, None]


def test_rule_check_error_codes_without_gpu(handle):
    f, one = handle.tb_rule_check, 16
    for k in PTRS:
        assert f(*_args(one, **{k: None})) == TB_ERR_NULL, k
    for k in DIMS:
        for v in (0, -1):
            assert f(*_args(one, **{k: v})) == TB_ERR_BAD_SHAPE, (k, v)
    assert f(*_args(one, A=RS.MAX_A + 1)) == TB_ERR_UNSUPPORTED
    assert f(*_args(None, A=RS.MAX_A + 1)) == TB_ERR_NULL  # pointers are checked first


@pytest.mark.parametrize("name", sorted(RS.BUILDERS))
def test_scene_fp32_oracle_agrees_with_float64(name):
    s = RS.BUILDERS[name]()
    f64, c64 = RS.replay(s)
    f32, c32 = RS.replay(s, torch.float32)
    for k in RS.VIO:
        assert torch.equal(f64[k], f32[k]), k
    assert torch.equal(c64, c32)


@pytest.mark.parametrize("name", ["pairs", "road_edge", "red_light", "passive", "single_agent"])
def test_hand_placed_cases_have_their_pattern(name):
    s = RS.BUILDERS[name]()
    ref, _ = RS.replay(s)
    assert s.expect
    for b, a, flag, want in s.expect:
        assert torch.equal(ref[flag][b, a], want), (b, a, flag, ref[flag][b, a].tolist(), want.tolist())
    if name == "pairs":  # corner contacts: collided without collided_wosac; pedestrian pairs: the other way round
        col, wos = ref["collided"], ref["collided_wosac"]
        assert bool((col & ~wos).any()) and bool((wos & ~col).any())
    if name == "passive":  # the counter passes 20 at the 21st consecutive passive step
        assert int(ref["passive"][..., :20].sum()) == 0 and bool(ref["passive"][..., 20].any())
    if name == "single_agent":
        assert s.pred_valid.shape[1] == 1


def test_crowd_overflows_the_pair_queue_with_mixed_outcomes():
    s = RS.crowd()
    assert s.pred_valid.shape[1] == RS.MAX_A
    assert int(RS.pair_queue_count(s).min()) > RS.QCAP
    ref, _ = RS.replay(s)
    valid = s.pred_valid
    col = ref["collided"][valid].float().mean()
    assert 0.2 <= float(col) <= 0.8, float(col)
    assert bool((ref["collided"] != ref["collided_wosac"]).any())


def test_dense_map_overflows_the_map_queue():
    s = RS.dense_map()
    assert int(RS.map_queue_count(s).min()) > RS.QCAP
    ref, _ = RS.replay(s)
    assert bool(ref["run_road_edge"].any()) and not bool(ref["run_road_edge"].all())
    # lane-centre nodes within 2 m of vehicles (the passive check's lane proximity) are among the queued pairs too
    tab = RS.kernel_tables(s)
    lane_node = (tab["poly_kind"][:, :, None] & 2).bool() & ~tab["node_invalid"].bool()
    xy = s.pred_pose[0, :, 0, :2]
    d = (s.mp_pos[0][lane_node[0]][:, None] - xy[None]).norm(dim=-1)
    assert int((d < 2).any(0).sum()) > 0


def test_mixed_scenes_use_distinct_rows():
    """The engine-layout scenes give a different result when the map / TL rows are indexed by the rollout."""
    for s in (RS.mixed(), RS.mixed(tl_per_rollout=True)):
        ref, _ = RS.replay(s)
        B = s.pred_valid.shape[0]
        wrong = RS.SimpleNamespace(**vars(s))
        wrong.tl_state = s.tl_state[(torch.arange(B) // s.tl_div).flip(0)]
        wrong.tl_div = 1
        alt, _ = RS.replay(wrong)
        assert not torch.equal(ref["run_red_light"], alt["run_red_light"]) or \
            not torch.equal(ref["passive"], alt["passive"])
