"""GPU: caller control of the rollout engine — the player override in the dynamics step (tb_dyn_step_player), open-loop
plans, log replay of whole agents ("tf/forcing_agent") and step-by-step stepping (begin / step) — against the CPU
reference of tests/_player_oracle.py, and against the engine's own paths without players."""
import pytest
import torch

from trafficbotsv1_5_b200 import config, params, synth

import _player_oracle as PO

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from trafficbotsv1_5_b200 import lib as L, ops
    from trafficbotsv1_5_b200.engine import RolloutEngine

DEV = "cuda"
# closed-loop tolerances of tests/test_rollout_gpu.py: fp32 mode over the rollout; tensor-core mode (DESIGN.md 7)
TOL_XY, TOL_YAW = 5e-3, 1e-3
TC_TOL_XY, TC_TOL_YAW = 2e-2, 5e-3
GOLDEN_SHAPE = dict(n_sc=2, n_ag=32, n_mp=96, n_tl=30, seed=1000, boundary=105.0)  # tests/golden/rollout_small.pt
MASKS = ("pred_valid", "tl_state", "final_valid", "final_navi_valid")


def maxerr(a, b):
    return float((a.detach().float().cpu() - b.detach().float().cpu()).abs().max())


def _setup(shape, R, T, **kw):
    cfg = config.default_model_cfg()
    P = params.init_params(cfg, seed=0)
    return RolloutEngine(P, cfg, DEV, n_rollout=R, step_end=T, **kw), synth.make_scene_batch(**shape), P, cfg


def _oracle(P, cfg, batch, R, T, **kw):
    return PO.rollout(P, cfg, config.derived_sizes(cfg), config.DYNAMICS_CFG, config.ROLLOUT_CFG, batch, R, T, **kw)


def _clone(res):
    return {k: v.clone() for k, v in res.items() if torch.is_tensor(v)}


def _same_bits(a, b, keys=("pred_valid", "pred_pose", "pred_motion", "tl_state", "final_valid", "final_navi_valid")):
    for k in keys:
        assert torch.equal(a[k], b[k]), k


def _compare(res, ref, precision, what=""):
    for k in MASKS:
        n = int((res[k].cpu() != ref[k]).sum())
        assert n == 0, f"{what}{k}: {n} mismatches"
    e_xy = maxerr(res["pred_pose"][..., :2], ref["pred_pose"][..., :2])
    e_yaw = maxerr(res["pred_pose"][..., 2], ref["pred_pose"][..., 2])
    print(f"{what}precision={precision}: xy {e_xy:.2e} m, yaw {e_yaw:.2e} rad")
    assert e_xy < (TC_TOL_XY if precision else TOL_XY) and e_yaw < (TC_TOL_YAW if precision else TOL_YAW)


def _plan(batch, R, T, n_players=2, per_rollout=True, seed=0):
    """Players: the first `n_players` agents of every scene that are valid at t = 0 and have a type; per rollout a
    different smooth plan (acc in [-2, 2] m/s^2, yaw rate up to 0.15 rad/s)."""
    n_sc, A, _ = batch["sc/ag_valid"].shape
    ok = batch["sc/ag_valid"][:, :, 0] & batch["ref/ag_type"].any(-1)
    pv = torch.zeros(n_sc, A, dtype=torch.bool)
    for sc in range(n_sc):
        pv[sc, torch.nonzero(ok[sc])[:n_players, 0]] = True
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(T, dtype=torch.float32)
    amp = torch.rand(n_sc, R, A, 1, generator=g) * 4 - 2
    ph = torch.rand(n_sc, R, A, 1, generator=g) * 6.28
    acc = amp * torch.cos(0.2 * t + ph)
    yr = 0.15 * torch.sin(0.1 * t + ph) * torch.sign(amp)
    pa = torch.stack([acc, yr], -1)                                       # [n_sc, R, A, T, 2]
    return pv, (pa if per_rollout else pa[:, 0].contiguous())


def _with(batch, **kv):
    out = dict(batch)
    out.update({k.replace("__", "/"): v for k, v in kv.items()})
    return out


# ---------------------------------------------------------------------------------------------- kernel
def _dyn_state(seed=0, n_sc=2, R=3, A=37, T=8, n_gt=10, W=11, n_mp=5, n_node=4, s=3):
    """Random tb_dyn_step inputs with invalid agents, agents without a type, forced, disabled and out-of-map agents."""
    g = torch.Generator().manual_seed(seed)
    B = n_sc * R
    rnd = lambda *sh: torch.rand(*sh, generator=g)  # noqa: E731
    typ = torch.randint(0, 4, (B, A), generator=g)                       # 3: no type
    ag_type = torch.zeros(B, A, 3, dtype=torch.uint8)
    for t in range(3):
        ag_type[..., t] = (typ == t).to(torch.uint8)
    st = dict(
        act_branch=torch.randn(B * A, 6, generator=g), ag_type=ag_type,
        valid=(rnd(B, A) < 0.8).to(torch.uint8), disabled=(rnd(B, A) < 0.1).to(torch.uint8),
        navi_invalid=torch.zeros(B, A, dtype=torch.uint8), dest_reached=(rnd(B, A) < 0.2).to(torch.uint8),
        pose=torch.randn(B, A, 3, generator=g) * torch.tensor([30.0, 30.0, 2.0]),
        motion=torch.randn(B, A, 3, generator=g) * 5,
        gt_valid=(rnd(n_sc, A, n_gt) < 0.7).to(torch.uint8),
        gt_pose=torch.randn(n_sc, A, n_gt, 3, generator=g) * 20, gt_motion=torch.randn(n_sc, A, n_gt, 3, generator=g),
        boundary=torch.tensor([[-40.0, 40.0, -40.0, 40.0]]).repeat(n_sc, 1),
        dest_idx=torch.randint(0, n_mp, (B, A), generator=g, dtype=torch.int32),
        mp_pos=torch.randn(n_sc, n_mp, n_node, 2, generator=g) * 30,
        mp_dirn=torch.nn.functional.normalize(torch.randn(n_sc, n_mp, n_node, 2, generator=g), dim=-1),
        mp_node_invalid=(rnd(n_sc, n_mp, n_node) < 0.2).to(torch.uint8),
        mp_kind=torch.randint(0, 3, (n_sc, n_mp), generator=g, dtype=torch.uint8),
        d_step=torch.tensor([s], dtype=torch.int32),
        hist_valid=torch.zeros(B, A, W, dtype=torch.uint8), hist_pose=torch.zeros(B, A, W, 3),
        hist_motion=torch.zeros(B, A, W, 3), pred_valid=torch.zeros(B, A, T, dtype=torch.uint8),
        pred_pose=torch.zeros(B, A, T, 3), pred_motion=torch.zeros(B, A, T, 3),
        o_outside=torch.zeros(B, A, T, dtype=torch.uint8), o_reached=torch.zeros(B, A, T, dtype=torch.uint8))
    st["tf_mask"] = st["gt_valid"] * (rnd(n_sc, A, n_gt) < 0.5).to(torch.uint8)
    st["pose"][:, :3, 0] = 39.99                                         # on the map edge: players may leave it
    st = {k: v.to(DEV).contiguous() for k, v in st.items()}
    return st, dict(n_sc=n_sc, R=R, B=B, A=A, T=T, n_gt=n_gt, W=W, n_mp=n_mp, n_node=n_node, s=s)


def _launch(st, d, player_valid=None, player_action=None, entry="tb_dyn_step_player"):
    dy = config.DYNAMICS_CFG
    order = ("veh", "ped", "cyc")
    args = [L.ptr(st["act_branch"]), L.ptr(st["ag_type"]), ops.host_f3([dy[k]["max_acc"] for k in order]),
            ops.host_f3([dy[k]["max_yaw_rate"] for k in order]), dy["dt"], L.ptr(st["valid"]), L.ptr(st["disabled"]),
            L.ptr(st["navi_invalid"]), L.ptr(st["dest_reached"]), L.ptr(st["pose"]), L.ptr(st["motion"]),
            L.ptr(st["gt_valid"]), L.ptr(st["gt_pose"]), L.ptr(st["gt_motion"]), L.ptr(st["tf_mask"]), d["n_gt"], d["R"],
            L.ptr(st["boundary"]), L.ptr(st["dest_idx"]), L.ptr(st["mp_pos"]), L.ptr(st["mp_dirn"]),
            L.ptr(st["mp_node_invalid"]), L.ptr(st["mp_kind"]), d["n_mp"], d["n_node"], 50.0, 10.0, 0.866,
            L.ptr(st["d_step"]), d["B"], d["A"], d["W"], d["T"], L.ptr(st["hist_valid"]), L.ptr(st["hist_pose"]),
            L.ptr(st["hist_motion"]), L.ptr(st["pred_valid"]), L.ptr(st["pred_pose"]), L.ptr(st["pred_motion"]),
            L.ptr(st["o_outside"]), L.ptr(st["o_reached"])]
    if entry == "tb_dyn_step_player":
        args += [L.ptr(player_valid), L.ptr(player_action)]
    L.check(getattr(L.load(), entry)(*args, L.stream()), entry)
    torch.cuda.synchronize()


def test_kernel_without_players_matches_dyn_step_ex():
    for seed in range(3):
        st0, d = _dyn_state(seed)
        ref = {k: v.clone() for k, v in st0.items()}
        _launch(ref, d, entry="tb_dyn_step_ex")
        pa = torch.randn(d["B"] * d["A"], d["T"], 2, device=DEV) * 5
        for pv in (None, torch.zeros(d["B"] * d["A"], dtype=torch.uint8, device=DEV)):
            out = {k: v.clone() for k, v in st0.items()}
            _launch(out, d, pv, None if pv is None else pa)
            for k in out:
                assert torch.equal(out[k], ref[k]), (seed, k)
        assert int(ref["o_outside"].sum()) > 0 and int((st0["valid"] == 0).sum()) > 0


def test_kernel_with_players_vs_oracle():
    st0, d = _dyn_state(7)
    B, A, T, s = d["B"], d["A"], d["T"], d["s"]
    sc = torch.arange(B, device=DEV) // d["R"]
    forced = (st0["tf_mask"][sc, :, s] != 0) & (st0["disabled"] == 0)
    valid, typed = st0["valid"] != 0, (st0["ag_type"] != 0).any(-1)
    g = torch.Generator(device=DEV).manual_seed(3)
    pv = torch.rand(B, A, device=DEV, generator=g) < 0.5
    # a player on a forced agent (teacher forcing wins) and one on an invalid agent (no effect)
    i_forced = torch.nonzero(forced & valid & typed)[0]
    i_invalid = torch.nonzero(~valid)[0]
    pv[i_forced[0], i_forced[1]] = pv[i_invalid[0], i_invalid[1]] = True
    pa = torch.randn(B, A, T, 2, device=DEV, generator=g) * 4
    out = {k: v.clone() for k, v in st0.items()}
    _launch(out, d, pv.to(torch.uint8).contiguous(), pa.contiguous())
    # the oracle: policy action of the agent's type branch, then the override, then the unicycle update
    type_idx = st0["ag_type"].float().argmax(-1)
    br = st0["act_branch"].view(B, A, 3, 2)
    mean = torch.gather(br, 2, type_idx[..., None, None].expand(-1, -1, 1, 2))[:, :, 0]
    c = lambda t: t.cpu()  # noqa: E731
    p_ref, m_ref = PO.dynamics_update(c(st0["pose"]), c(st0["motion"]), c(valid), c(st0["ag_type"] != 0), c(mean),
                                      config.DYNAMICS_CFG, c(pv), c(pa[:, :, s - 1]))
    assert maxerr(out["pred_pose"][:, :, s - 1], p_ref) < 1e-5 and maxerr(out["pred_motion"][:, :, s - 1], m_ref) < 1e-5
    assert torch.equal(out["pred_valid"][:, :, s - 1], st0["valid"])
    on = pv & valid & typed
    assert torch.equal(out["pred_motion"][:, :, s - 1, 1:][on], pa[:, :, s - 1][on])
    # teacher forcing overrides the player: state = ground truth bits
    a = i_forced
    assert torch.equal(out["pose"][a[0], a[1]], st0["gt_pose"][sc[a[0]], a[1], s])
    assert not torch.equal(out["pred_pose"][a[0], a[1], s - 1], st0["gt_pose"][sc[a[0]], a[1], s])
    # the invalid player agent: zeros, no effect
    a = i_invalid
    assert float(out["pred_pose"][a[0], a[1], s - 1].abs().max()) == 0.0
    # state bookkeeping after the prediction: teacher forcing, disable outside the map unless the ground truth is valid
    pp = p_ref.to(DEV)
    bd = st0["boundary"][sc]
    outside = valid & ((pp[..., 0] > bd[:, None, 1]) | (pp[..., 0] < bd[:, None, 0]) | (pp[..., 1] > bd[:, None, 3])
                       | (pp[..., 1] < bd[:, None, 2]))
    assert torch.equal(out["o_outside"][:, :, s - 1] != 0, outside) and bool((outside & pv).any())
    gtv = st0["gt_valid"][sc, :, s] != 0
    dis = outside & ~gtv
    v_new = (valid | forced) & ~dis
    assert torch.equal(out["valid"] != 0, v_new)
    assert torch.equal(out["disabled"] != 0, (st0["disabled"] != 0) | dis)
    assert maxerr(out["pose"][~forced], pp[~forced]) < 1e-5
    assert torch.equal(out["pose"][forced], st0["gt_pose"][sc, :, s][forced])
    assert torch.equal(out["motion"][forced], st0["gt_motion"][sc, :, s][forced])


# ---------------------------------------------------------------------------------------------- engine vs oracle
_REF = {}


def _oracle_cached(key, P, cfg, batch, R, T, **kw):
    if key not in _REF:
        _REF[key] = _oracle(P, cfg, batch, R, T, **kw)
    return _REF[key]


@pytest.mark.parametrize("R", [2, 32])
@pytest.mark.parametrize("precision", [0, 1])
def test_open_loop_plan_vs_oracle(R, precision):
    T = 24
    eng, batch, P, cfg = _setup(GOLDEN_SHAPE, R, T, precision=precision)
    pv, pa = _plan(batch, R, T)
    res = _clone(eng.rollout(_with(batch, player__valid=pv, player__action=pa)))
    ref = _oracle_cached(("plan", R), P, cfg, batch, R, T,
                         player=lambda s, v, p, m: (pv.repeat_interleave(R, 0), pa.reshape(-1, pa.shape[2], T, 2)[:, :, s - 1]))
    _compare(res, ref, precision, f"plan R={R} ")
    # every valid step of a player records its plan's action bits, and the plan moved the players
    rows = pv.repeat_interleave(R, 0).to(DEV)
    plan = pa.reshape(-1, pa.shape[2], T, 2).to(DEV)
    on = res["pred_valid"][rows]
    assert torch.equal(res["pred_motion"][rows][..., 1:][on], plan[rows][on]) and int(on.sum()) > 0
    plain = eng.rollout(batch)
    assert maxerr(plain["pred_pose"][rows], res["pred_pose"][rows]) > 0.05


def test_log_replay_vs_oracle():
    R, T = 3, 24
    shape = dict(GOLDEN_SHAPE, n_hist=30)                              # ground truth beyond the warm start
    eng, batch, P, cfg = _setup(shape, R, T)
    n_sc, A, _ = batch["sc/ag_valid"].shape
    fa = torch.zeros(n_sc, A, dtype=torch.bool)
    fa[:, :8] = True
    b = _with(batch, tf__forcing_agent=fa)
    res = _clone(eng.rollout(b))
    ref = _oracle(P, cfg, batch, R, T, forcing_agent=fa)
    _compare(res, ref, 0, "log replay ")
    # step by step: forced agents sit exactly on their ground truth wherever it is valid
    obs = eng.begin(b)
    gt_v, gt_p = batch["sc/ag_valid"].to(DEV), batch["sc/ag_pose"].to(DEV)
    rows = fa.repeat_interleave(R, 0).to(DEV)
    n_checked = 0
    while True:
        t = obs["t"]
        on = rows & gt_v.repeat_interleave(R, 0)[:, :, t]
        assert torch.equal(obs["pose"][on], gt_p.repeat_interleave(R, 0)[:, :, t][on]), t
        assert bool(obs["valid"][on].all())
        n_checked += int(on.sum())
        if t == T:
            break
        obs = eng.step()
    assert n_checked > 0
    _same_bits(eng.results(), res)


def _controller(R, v_target0=4.0):
    """acc = 2 tanh(v_target - v), yaw rate 0; v_target differs per rollout. Works on CPU and GPU tensors."""
    def ctrl(step, valid, pose, motion):
        B = valid.shape[0]
        v_t = v_target0 + 2.0 * (torch.arange(B, device=motion.device) % R).to(motion.dtype)
        acc = 2.0 * torch.tanh(v_t[:, None] - motion[..., 0])
        return ctrl.pv.to(valid.device), torch.stack([acc, torch.zeros_like(acc)], -1)
    return ctrl


def test_closed_loop_controller_vs_oracle():
    R, T = 2, 24
    eng, batch, P, cfg = _setup(GOLDEN_SHAPE, R, T)
    eng.warm_dedup = False                                             # every step goes through step() and the controller
    n_sc, A, _ = batch["sc/ag_valid"].shape
    pv, _ = _plan(batch, R, T, n_players=3)
    ctrl = _controller(R)
    ctrl.pv = pv.repeat_interleave(R, 0)
    obs = eng.begin(_with(batch, player__valid=pv))
    assert obs["t"] == 0
    while obs["t"] < T:
        _, act = ctrl(obs["t"] + 1, obs["valid"], obs["pose"], obs["motion"])
        obs = eng.step(act.view(n_sc, R, A, 2))
    res = _clone(eng.results())
    ref = _oracle(P, cfg, batch, R, T, player=ctrl)
    _compare(res, ref, 0, "closed loop ")
    rows = ctrl.pv.to(DEV)
    assert float(res["pred_motion"][rows][:, -1, 0].sub(res["pred_motion"][rows][:, 0, 0]).abs().max()) > 0.1


@pytest.mark.parametrize("use_graph", [True, False])
def test_step_with_fixed_plan_equals_run(use_graph):
    R, T = 3, 24
    eng, batch, P, cfg = _setup(GOLDEN_SHAPE, R, T, use_graph=use_graph)
    pv, pa = _plan(batch, R, T)
    b = _with(batch, player__valid=pv, player__action=pa)
    ref = _clone(eng.rollout(b))
    obs = eng.begin(_with(batch, player__valid=pv, player__action=pa))
    assert obs["t"] == eng._s0 > 0                                     # warm start de-duplicated
    while obs["t"] < T:
        obs = eng.step(pa[:, :, :, obs["t"]])
    _same_bits(eng.results(), ref)
    # and from a zero plan, every column supplied by step(), without de-duplication
    eng.warm_dedup = False
    obs = eng.begin(_with(batch, player__valid=pv))
    while obs["t"] < T:
        obs = eng.step(pa[:, :, :, obs["t"]])
    eng.warm_dedup = True
    _same_bits(eng.results(), ref, keys=MASKS)
    assert maxerr(eng.results()["pred_pose"], ref["pred_pose"]) < 1e-4


# ---------------------------------------------------------------------------------------------- fast paths
@pytest.mark.parametrize("precision", [0, 1])
def test_players_warm_dedup_on_off(precision):
    R, T = 3, 24
    eng, batch, P, cfg = _setup(dict(n_sc=2, n_ag=40, n_mp=96, n_tl=30, seed=77, boundary=110.0), R, T, precision=precision)
    pv, pa = _plan(batch, R, T, n_players=3)
    b = _with(batch, player__valid=pv, player__action=pa)
    eng.prepare(b)
    assert eng._s0 == 11
    a = _clone(eng.run())
    eng.warm_dedup = False
    eng.prepare(b)
    assert eng._s0 == 0
    c = eng.run()
    _same_bits(a, c, keys=MASKS)
    tol = 1e-4 if precision == 0 else 2e-3
    assert maxerr(a["pred_pose"], c["pred_pose"]) < tol and maxerr(a["pred_motion"], c["pred_motion"]) < 5 * tol


@pytest.mark.parametrize("precision", [0, 1])
def test_players_compaction_on_off(precision):
    R, T = 3, 20
    eng, batch, P, cfg = _setup(dict(n_sc=2, n_ag=64, n_mp=96, n_tl=30, seed=91, boundary=110.0), R, T,
                                precision=precision, record_feedback=True)
    batch["sc/ag_valid"][:, 40:] = False
    batch["sc/ag_valid"][0, 3] = False                                  # holes next to player agents 2 and 4
    batch["sc/ag_valid"][1, 7] = False
    batch["ag_navi_valid"] = batch["ag_latent_valid"] = batch["sc/ag_valid"].any(-1)
    pv = torch.zeros(2, 64, dtype=torch.bool)
    pv[0, [2, 4]] = pv[1, [6, 8]] = True
    pv[0, 50] = True                                                    # a player on a dropped slot: never valid
    _, pa = _plan(batch, R, T, seed=4)
    b = _with(batch, player__valid=pv, player__action=pa, tf__forcing_agent=torch.arange(64)[None].expand(2, -1) == 10)
    eng.prepare(b)
    assert eng._perm is not None and eng._st["A"] < 44
    a = _clone(eng.run())
    eng.compact_agents = False
    eng.prepare(b)
    assert eng._perm is None
    c = eng.run()
    _same_bits(a, c, keys=MASKS + ("outside_map", "dest_reached"))
    # 1e-5 m (fp32) as in test_agent_compaction_matches_padded_run, but at least 2 ulp of the largest coordinate: the
    # GEMM row tiling re-rounds, and these players travel to ~75 m where 2 ulp of fp32 are 1.5e-5 m
    ulp2 = 2 * torch.finfo(torch.float32).eps * float(c["pred_pose"][..., :2].abs().max())
    tol = max(1e-5, ulp2) if precision == 0 else 2e-3
    assert maxerr(a["pred_pose"], c["pred_pose"]) < tol, (maxerr(a["pred_pose"], c["pred_pose"]), tol)
    never = ~batch["sc/ag_valid"].any(-1).repeat_interleave(R, 0).to(DEV)
    assert float(a["pred_pose"][never].abs().max()) == 0.0


def test_graphs_alternate_with_and_without_players():
    R, T = 2, 20
    shape = dict(n_sc=2, n_ag=40, n_mp=96, n_tl=30, seed=93, boundary=110.0)
    eng, batch, P, cfg = _setup(shape, R, T, precision=1)
    pv, pa = _plan(batch, R, T)
    with_p = _with(batch, player__valid=pv, player__action=pa)
    fresh = {}
    for name, b in (("plain", batch), ("players", with_p)):
        e2, _, _, _ = _setup(shape, R, T, precision=1)
        fresh[name] = _clone(e2.rollout(b))
    assert maxerr(fresh["plain"]["pred_pose"], fresh["players"]["pred_pose"]) > 0.01
    graphs = {}
    for name, b in (("plain", batch), ("players", with_p)) * 2:
        out = eng.rollout(b)
        _same_bits(out, fresh[name])
        graphs.setdefault(name, eng._graph)
        assert eng._graph is graphs[name]
    assert graphs["plain"] is not graphs["players"]
    # no player at all in "player/valid": the bits of the batch without the keys
    empty = _with(batch, player__valid=torch.zeros_like(pv), player__action=pa)
    _same_bits(eng.rollout(empty), fresh["plain"])
    _same_bits(eng.rollout(_with(batch, tf__forcing_agent=torch.zeros_like(pv))), fresh["plain"])


def test_input_checks():
    R, T = 2, 12
    eng, batch, P, cfg = _setup(dict(n_sc=1, n_ag=30, n_mp=80, n_tl=28, seed=9, boundary=110.0), R, T)
    pv, pa = _plan(batch, R, T)
    bad = [dict(player__valid=pv),                                          # no plan
           dict(player__action=pa),                                         # plan without players
           dict(player__valid=pv.float(), player__action=pa),
           dict(player__valid=pv[:, :-1], player__action=pa),
           dict(player__valid=pv, player__action=pa[..., :-1, :]),          # not step_end columns
           dict(player__valid=pv, player__action=pa[:, :1].expand(-1, 3, -1, -1, -1)),   # R = 3 plans for R = 2
           dict(player__valid=pv, player__action=torch.where(torch.arange(T) == 5, float("nan"), 0.0)[:, None]
                .expand(*pa.shape[:-1], 2) + pa),
           dict(player__valid=pv, player__action=pa.clone().index_fill_(3, torch.tensor([2]), float("inf"))),
           dict(tf__forcing_agent=pv.float()),
           dict(tf__forcing_agent=pv[:, :5])]
    for kv in bad:
        with pytest.raises(ValueError):
            eng.prepare(_with(batch, **kv))
    with pytest.raises(RuntimeError):
        eng.step(pa[:, :, :, 0])                                            # not begun
    eng.begin(_with(batch, player__valid=pv))
    with pytest.raises(ValueError):
        eng.step(pa[:, :, :-1, 0])
    with pytest.raises(ValueError):
        eng.step(torch.full_like(pa[:, :, :, 0], float("nan")))
    eng.begin(batch)
    with pytest.raises(ValueError):
        eng.step(pa[:, :, :, 0])                                            # the batch has no players
    while eng._t < T:
        eng.step()
    with pytest.raises(RuntimeError):
        eng.step()
