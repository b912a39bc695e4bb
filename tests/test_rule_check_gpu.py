"""tb_rule_check (csrc/rule_check.cu) flag for flag against the float64 replay of the oracle's RuleCheckOracle on the
scenes of tests/_rule_scenes.py: hand-placed pairs, road edges, red lights and passive vehicles, both queue-overflow
paths (an A = 256 crowd and a dense map), A = 1, the engine's layout (div = tl_div = R) and the per-rollout TL layout,
steps past the history ring, and steps outside [1, T]. Then the engine's own flags on a rule-check scene."""
import gc

import pytest
import torch

import _rule_scenes as RS
from oracle import tb_oracle as O
from trafficbotsv1_5_b200 import config, params, synth

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _decoy(state):
    """A contradicting one-hot state: 3 (neither red nor blocking) for 0/1/2/4, red for 3."""
    k = state.to(torch.uint8).argmax(-1)
    return torch.nn.functional.one_hot(torch.where(k == 3, RS.RED, 3), 5).to(torch.uint8)


def run_kernel(s, steps=None, counter0=None, outs0=None):
    """tb_rule_check for steps 1..T (or `steps`) the way the engine calls it. The hist_tl ring has B rows (only the first
    B / tl_div belong to the layout); before step s slot s % W of those rows holds the step's TL state, and every other
    slot and row holds a contradicting state, so reading a wrong slot or row changes flags."""
    from trafficbotsv1_5_b200 import lib as L
    B, A, T = s.pred_valid.shape
    n_tl = s.tl_valid.shape[1]
    Bt = s.tl_state.shape[0]
    d = lambda t, dt=None: t.to(DEV, dt).contiguous()  # noqa: E731
    tab = {k: d(v) for k, v in RS.kernel_tables(s).items()}
    pv, pp, pm = d(s.pred_valid, torch.uint8), d(s.pred_pose), d(s.pred_motion)
    ag_type, ag_size = d(s.ag_type, torch.uint8), d(s.ag_size)
    tl_inv, tl_pose = d(~s.tl_valid, torch.uint8), d(s.tl_pose)
    tl_state = d(s.tl_state, torch.uint8)
    hist_tl = torch.zeros(B, n_tl, RS.W, 5, dtype=torch.uint8, device=DEV)
    counter = torch.zeros(B, A, device=DEV) if counter0 is None else d(counter0)
    outs = {k: torch.zeros(B, A, T, dtype=torch.uint8, device=DEV) if outs0 is None else d(outs0[k]) for k in RS.VIO}
    d_step = torch.zeros(1, dtype=torch.int32, device=DEV)
    pad = torch.arange(B, device=DEV) % Bt
    for st in (range(1, T + 1) if steps is None else steps):
        t = min(max(st, 1), T) - 1
        hist_tl.copy_(_decoy(tl_state[pad, :, t])[:, :, None].expand(-1, -1, RS.W, -1))
        hist_tl[:Bt, :, st % RS.W] = tl_state[:, :, t]
        d_step.fill_(st)
        L.check(L.load().tb_rule_check(
            L.ptr(pv), L.ptr(pp), L.ptr(pm), L.ptr(ag_type), L.ptr(ag_size), L.ptr(hist_tl), L.ptr(tl_inv),
            L.ptr(tl_pose), L.ptr(tab["seg"]), L.ptr(tab["node_invalid"]), L.ptr(tab["poly_circle"]),
            L.ptr(tab["poly_kind"]), tab["seg"].shape[1], tab["seg"].shape[2], L.ptr(counter),
            *[L.ptr(outs[k]) for k in RS.VIO], L.ptr(d_step), B, A, T, RS.W, n_tl, s.div, s.tl_div, RS.SIZE_SCALE,
            L.stream()), "tb_rule_check")
    torch.cuda.synchronize()
    return {k: v.bool().cpu() for k, v in outs.items()}, counter.cpu()


def _assert_exact(s):
    mine, counter = run_kernel(s)
    ref, ref_counter = RS.replay(s)
    for k in RS.VIO:
        diff = (mine[k] != ref[k]).nonzero().tolist()
        assert not diff, f"{k}: {len(diff)} (rollout, agent, step) differ from the float64 reference, first {diff[:5]}"
    assert torch.equal(counter, ref_counter.float()), "passive_counter"
    return ref


@pytest.mark.parametrize("name", ["pairs", "road_edge", "red_light", "passive", "single_agent", "crowd", "dense_map",
                                  "mixed_per_scene", "mixed_per_rollout"])
def test_rule_check_exact_vs_float64(name):
    s = RS.BUILDERS[name]()
    ref = _assert_exact(s)
    if name == "crowd":      # the pair queue overflowed: the pairs past QCAP were tested inline
        assert s.pred_valid.shape[1] == RS.MAX_A and int(RS.pair_queue_count(s).min()) > RS.QCAP
    if name == "dense_map":  # the (polyline, vehicle) queue overflowed
        assert int(RS.map_queue_count(s).min()) > RS.QCAP and bool(ref["run_road_edge"].any())
    if name.startswith("mixed"):
        assert s.div > 1 and s.T > RS.W and all(int(ref[k].sum()) > 0 for k in RS.VIO)


@pytest.mark.parametrize("step", [0, -1, "T+1", "T+7"])
def test_rule_check_steps_outside_range_write_nothing(step):
    """d_step outside [1, T]: the flag buffers and the passive counter come back byte for byte."""
    s = RS.passive()
    B, A, T = s.pred_valid.shape
    st = T + int(step[2:]) if isinstance(step, str) else step
    outs0 = {k: torch.full((B, A, T), 0xA5, dtype=torch.uint8) for k in RS.VIO}
    counter0 = torch.full((B, A), 7.25)
    mine, counter = run_kernel(s, steps=[st], counter0=counter0, outs0=outs0)
    for k in RS.VIO:
        assert bool((mine[k] == (outs0[k] != 0)).all())
    assert torch.equal(counter, counter0)


def test_rule_check_counter_carries_across_calls():
    """Steps 1..T in two runs of calls (1..12, then 13..T on the returned counter and flags) equal one run."""
    s = RS.passive()
    a, ca = run_kernel(s)
    T = s.T
    b1, cb = run_kernel(s, steps=range(1, 13))
    b, cb = run_kernel(s, steps=range(13, T + 1), counter0=cb, outs0={k: v.to(torch.uint8) for k, v in b1.items()})
    assert torch.equal(ca, cb) and all(torch.equal(a[k], b[k]) for k in RS.VIO)


# ---------------------------------------------------------------------------------------------- engine level
@pytest.mark.parametrize("compact", [True, False])
def test_engine_rule_checks_vs_oracle_on_engine_trajectories(compact):
    """RolloutEngine(rule_checks=True) at n_sc = 2, R = 3 on a scene where red light and passive fire; the oracle is
    replayed on the engine's own pred_* and TL states, so trajectory drift does not enter the comparison. These are
    closed-loop trajectories (no jitter filter), so knife-edge cases keep the usual budget: <= max(1, 0.5 %) of the
    positives of each flag."""
    from trafficbotsv1_5_b200.engine import RolloutEngine
    gc.collect()  # graphs of an earlier engine kept alive by a failed test's traceback must not be freed during capture
    n_sc, R, T = 2, 3, 36
    cfg = config.default_model_cfg()
    eng = RolloutEngine(params.init_params(cfg, seed=0), cfg, DEV, n_rollout=R, step_end=T, rule_checks=True)
    eng.compact_agents = compact
    batch = synth.make_rule_scene_batch(n_sc=n_sc, n_ag=48, n_mp=96, n_tl=40, seed=5000)
    for k in ("sc/ag_valid", "ag_navi_valid", "ag_latent_valid"):  # never-valid slots: compaction drops them
        batch[k][:, 40:] = False
    res = {k: v.cpu() for k, v in eng.rollout(batch).items() if torch.is_tensor(v)}
    assert (eng._perm is not None) == compact
    rep = lambda t: t.repeat_interleave(R, 0)  # noqa: E731
    oc = O.RuleCheckOracle(rep(batch["map/valid"]), rep(batch["map/type"]), rep(batch["map/pos"][..., :2]),
                           rep(batch["map/dir"][..., :2]), rep(batch["ref/ag_type"]), rep(batch["ref/ag_size"]),
                           rep(batch["sc/tl_valid"]), rep(batch["sc/tl_pose"]))
    ref = {k: [] for k in RS.VIO}
    for t in range(T):
        for k, v in oc.check(res["pred_valid"][:, :, t], res["pred_pose"][:, :, t], res["pred_motion"][:, :, t],
                             res["tl_state"][:, :, t]).items():
            ref[k].append(v)
    for k in RS.VIO:
        r = torch.stack(ref[k], 2)
        n_diff, n_pos = int((res[k] != r).sum()), int(r.sum())
        print(f"{k}: oracle positives {n_pos}, mismatches {n_diff}")
        assert n_diff <= max(1, int(0.005 * n_pos)), f"{k}: {n_diff} mismatches of {n_pos} positives"
        if k in ("run_red_light", "passive"):
            assert n_pos >= 100, f"{k}: only {n_pos} positives"
