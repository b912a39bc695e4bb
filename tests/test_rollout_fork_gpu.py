"""GPU: snapshot / restore / fork of the rollout engine's step-by-step stepping (RolloutEngine.snapshot, .restore) and
the batched row copy behind them (tb_copy_rows). Unless noted: both precisions, rule checks and per-step feedback on,
agent compaction with holes in the agent axis, warm-start de-duplication on, per-rollout player plans."""
import pytest
import torch

from trafficbotsv1_5_b200 import config, params, synth

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from trafficbotsv1_5_b200 import ops
    from trafficbotsv1_5_b200.engine import RolloutEngine

DEV = "cuda"
SHAPE = dict(n_sc=2, n_ag=64, n_mp=96, n_tl=30, seed=91, boundary=110.0)


def _plan(batch, R, T, seed):
    """Per-rollout smooth plans for the agents 2, 4 (scene 0) and 6, 8 (scene 1), caller's agent order."""
    n_sc, A, _ = batch["sc/ag_valid"].shape
    pv = torch.zeros(n_sc, A, dtype=torch.bool)
    pv[0, [2, 4]] = pv[1, [6, 8]] = True
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(T, dtype=torch.float32)
    amp = torch.rand(n_sc, R, A, 1, generator=g) * 4 - 2
    ph = torch.rand(n_sc, R, A, 1, generator=g) * 6.28
    pa = torch.stack([amp * torch.cos(0.2 * t + ph), 0.15 * torch.sin(0.1 * t + ph) * torch.sign(amp)], -1)
    return pv, pa                                                       # [n_sc, A], [n_sc, R, A, T, 2]


def _setup(precision, R, T, use_graph=True, shared_latent=False):
    cfg = config.default_model_cfg()
    eng = RolloutEngine(params.init_params(cfg, seed=0), cfg, DEV, precision=precision, n_rollout=R, step_end=T,
                        rule_checks=True, record_feedback=True, use_graph=use_graph)
    b = synth.make_scene_batch(**SHAPE)
    b["sc/ag_valid"][:, 40:] = False                                    # padding dropped by agent compaction ...
    b["sc/ag_valid"][0, 3] = False                                      # ... and holes between kept slots
    b["sc/ag_valid"][1, 7] = False
    b["ag_navi_valid"] = b["ag_latent_valid"] = b["sc/ag_valid"].any(-1)
    if shared_latent:
        b["ag_latent"] = b["ag_latent"][:, :1].expand(-1, b["ag_latent"].shape[1], -1, -1).contiguous()
    pv, pa = _plan(b, R, T, seed=1)
    return eng, dict(b, **{"player/valid": pv, "player/action": pa}), pa


def _clone(d):
    return {k: (v.clone() if torch.is_tensor(v) else v) for k, v in d.items()}


def _same(a, b, what=""):
    assert a.keys() == b.keys(), (what, a.keys() ^ b.keys())
    for k in a:
        if torch.is_tensor(a[k]):
            assert a[k].shape == b[k].shape and torch.equal(a[k], b[k]), f"{what}{k}"
        else:
            assert a[k] == b[k], f"{what}{k}"


def _advance_to(eng, t, plan=None):
    obs = eng._observe()
    while obs["t"] < t:
        obs = eng.step(None if plan is None else plan[:, :, :, obs["t"]])
    return obs


def _fresh(eng, b, k, plan, H):
    """begin + steps up to k with the batch's plan + H steps with `plan` (None: the batch's plan); observations of
    the H steps and the results."""
    eng.begin(b)
    _advance_to(eng, k)
    obs = [_clone(eng.step(None if plan is None else plan[:, :, :, k + h])) for h in range(H)]
    return obs, _clone(eng.results())


# ---------------------------------------------------------------------------------------------- round trip
@pytest.mark.parametrize("precision", [0, 1])
def test_round_trip_is_exact(precision):
    R, T, H = 4, 24, 5
    eng, b, _ = _setup(precision, R, T)
    _, p1 = _plan(b, R, T, seed=11)
    _, p2 = _plan(b, R, T, seed=12)
    s0 = eng.begin(b)["t"]
    assert s0 > 0 and eng._perm is not None                              # warm start de-duplicated, agents compacted
    for k in (s0, s0 + 1, T - H):                                       # both TL buffer parities; a run to step_end
        ref_obs, ref = _fresh(eng, b, k, p2, H)
        ref_obs0, ref0 = _fresh(eng, b, k, None, H)
        eng.begin(b)
        at_k = _clone(_advance_to(eng, k))
        snap = eng.snapshot()
        assert snap.t == k
        for h in range(H):
            eng.step(p1[:, :, :, k + h])
        assert not torch.equal(eng.results()["pred_pose"], ref["pred_pose"])  # P1 went elsewhere
        _same(_clone(eng.restore(snap)), at_k, f"k={k} restore obs: ")
        for h in range(H):
            _same(_clone(eng.step(p2[:, :, :, k + h])), ref_obs[h], f"k={k} h={h} obs: ")
        _same(_clone(eng.results()), ref, f"k={k} P2: ")
        if k + H == T:
            with pytest.raises(RuntimeError):
                eng.step()
        # restore + step(None): the snapshot's plan columns (the batch's), not P2's
        eng.restore(snap)
        for h in range(H):
            _same(_clone(eng.step()), ref_obs0[h], f"k={k} h={h} plan obs: ")
        _same(_clone(eng.results()), ref0, f"k={k} plan: ")


# ---------------------------------------------------------------------------------------------- fork
@pytest.mark.parametrize("precision", [0, 1])
def test_fork_equals_run(precision):
    """The R rollouts of a scene share latent and destination and follow plans that agree before t_fork: their states
    at t_fork are equal, so forking any rollout into any other and continuing with the rollout's own plan must give
    the bits of run() with the full plans, rollout for rollout."""
    R, T = 4, 24
    eng, b, pa = _setup(precision, R, T, shared_latent=True)
    s0 = eng.begin(b)["t"]
    t_fork = s0 + 3
    pa = pa.clone()
    pa[:, :, :, :t_fork] = pa[:, :1, :, :t_fork]
    b["player/action"] = pa
    truth = _clone(eng.rollout(b))
    eng.begin(b)
    _advance_to(eng, t_fork)
    snap = eng.snapshot()
    src = torch.tensor([[3, 2, 1, 0], [1, 1, 3, 0]])                    # a reversal; duplicates and a dropped rollout
    obs = eng.restore(snap, src)
    assert obs["t"] == t_fork
    _advance_to(eng, T, pa)
    _same(_clone(eng.results()), truth, "fork: ")


@pytest.mark.parametrize("precision", [0, 1])
def test_fork_moves_exactly_the_state(precision):
    R, T = 4, 24
    eng, b, _ = _setup(precision, R, T)
    s0 = eng.begin(b)["t"]
    _advance_to(eng, s0 + 2)
    snap = eng.snapshot()
    _advance_to(eng, s0 + 4)                                            # the live state moved on
    st, d = eng._st, eng.model.d
    fixed = ["latent", "latent_invalid", "dest_idx", "ag_attr", "ag_type", "player_valid", "tf_mask", "gt_valid",
             "gt_pose", "gt_motion", "gt_tl", "init_navi_valid", "mp_pos", "mp_dirn", "boundary", "ag_size", "seg"]
    before = {k: st[k].clone() for k in fixed}
    navi = {"feat": eng._navi["feat"].clone(), "pose": eng._navi["pose"].clone(),
            "latent_cat": eng._navi["latent_cat"][:, d:].clone()}
    src = torch.tensor([[2, 2, 0, 1], [3, 0, 1, 1]], dtype=torch.int32)
    eng.restore(snap, src.to(DEV))
    items = eng._state_items()
    names = {k for k, _, pr in items if pr}
    assert {"valid", "pose", "hist_pose", "pred_pose", "knn_state", "knn_state_tl", "player_action", "passive_counter",
            "vio_collided", "fb_outside"} <= names
    n_sc = st["n_sc"]
    rows = (torch.arange(n_sc)[:, None] * R + src.long()).reshape(-1).to(DEV)
    for k, t, per_rollout in items:
        snap_t = snap._bufs[k]
        if per_rollout:
            if k in ("pose", "hist_pose", "pred_pose", "knn_state", "player_action"):
                assert not torch.equal(snap_t, snap_t[rows]), k         # rollouts differ: the gather moves rows
            assert torch.equal(t, snap_t[rows]), k
        else:
            assert torch.equal(t, snap_t), k
    for k in fixed:
        assert torch.equal(st[k], before[k]), k
    assert torch.equal(eng._navi["feat"], navi["feat"]) and torch.equal(eng._navi["pose"], navi["pose"])
    assert torch.equal(eng._navi["latent_cat"][:, d:], navi["latent_cat"])


# ---------------------------------------------------------------------------------------------- several snapshots, graphs
def test_nested_snapshots_in_any_order():
    R, T = 4, 24
    eng, b, _ = _setup(1, R, T)
    s0 = eng.begin(b)["t"]
    _, full = _fresh(eng, b, s0, None, T - s0)
    eng.begin(b)
    _advance_to(eng, s0 + 2)
    a = eng.snapshot()
    _advance_to(eng, s0 + 5)
    inner = eng.snapshot()
    _advance_to(eng, T)
    _same(_clone(eng.results()), full, "straight: ")
    for order in (("inner", "a"), ("a", "inner"), ("inner", "inner")):  # LIFO, non-LIFO, the same one twice
        for name in order:
            snap = inner if name == "inner" else a
            assert eng.restore(snap)["t"] == snap.t
            _advance_to(eng, T)
            _same(_clone(eng.results()), full, f"{order} {name}: ")


def test_players_and_plain_batches_keep_their_graphs():
    R, T = 4, 24
    eng, b, _ = _setup(1, R, T)
    plain = {k: v for k, v in b.items() if not k.startswith("player/")}
    ref = {}
    for name, bb in (("plain", plain), ("players", b)):
        eng.begin(bb)
        ref[name] = (_clone(_fresh(eng, bb, eng._t, None, T - eng._t)[1]), eng._graph)
    assert ref["plain"][1] is not ref["players"][1]
    for name, bb in (("players", b), ("plain", plain)) * 2:
        s0 = eng.begin(bb)["t"]
        _advance_to(eng, s0 + 3)
        snap = eng.snapshot()
        _advance_to(eng, T)
        eng.restore(snap, torch.arange(R).repeat(2, 1))                 # identity fork
        _advance_to(eng, T)
        assert eng._graph is ref[name][1]
        _same(_clone(eng.results()), ref[name][0], f"{name}: ")


def test_eager_matches_graph_path():
    R, T = 4, 24
    out = []
    for use_graph in (True, False):
        eng, b, pa = _setup(1, R, T, use_graph=use_graph)
        s0 = eng.begin(b)["t"]
        _advance_to(eng, s0 + 3)
        snap = eng.snapshot()
        _advance_to(eng, s0 + 6)
        eng.restore(snap, torch.tensor([[1, 0, 3, 3], [2, 2, 2, 2]]))
        assert eng._host_step == snap._host_step
        _advance_to(eng, T, pa)
        out.append(_clone(eng.results()))
    _same(out[0], out[1], "eager vs graph: ")


# ---------------------------------------------------------------------------------------------- the kernel alone
def _guarded(n_bytes, offset, dev=DEV):
    """A byte buffer with 64 guard bytes on both sides and a view of n_bytes starting `offset` bytes in."""
    buf = torch.randint(0, 256, (n_bytes + 128 + offset,), dtype=torch.uint8, device=dev)
    return buf, buf[64 + offset:64 + offset + n_bytes]


@pytest.mark.parametrize("dtype", [torch.uint8, torch.float16, torch.float32])
def test_copy_rows_kernel_vs_torch(dtype):
    g = torch.Generator(device=DEV).manual_seed(3)
    es = torch.tensor([], dtype=dtype).element_size()
    R = 4
    for width, n_sc, offset in ((1, 3, 0), (3, 2, 1), (37, 1, 0), (37, 40000, 1), (64, 5, 0), (64, 20000, 0),
                                (3, 30000, 0)):
        n_rows = n_sc * R
        row_bytes = width * es
        off = offset * es                                               # misaligned views: 1 element in
        items, keep = [], []
        for per_rollout in (True, False, True):
            sbuf, sb = _guarded(n_rows * row_bytes, off)
            dbuf, db = _guarded(n_rows * row_bytes, off)
            src, dst = sb.view(dtype).view(n_rows, width), db.view(dtype).view(n_rows, width)
            items.append((src, dst, per_rollout))
            keep.append((sbuf.clone(), dbuf.clone(), sbuf, dbuf))
        m = torch.randint(0, R, (n_rows,), generator=g, device=DEV, dtype=torch.int32)
        bad = torch.tensor([-1, R, 1000, -2**31, 2**31 - 1], dtype=torch.int32, device=DEV)
        m[: min(n_rows, 5)] = bad[: min(n_rows, 5)]                      # out of range: the row's own index
        m[-1] = -7
        ops.copy_rows(items, m, R)
        b = torch.arange(n_rows, device=DEV)
        ok = (m >= 0) & (m < R)
        rows = torch.where(ok, b - b % R + m.long().clamp(0, R - 1), b)
        for (src, dst, per_rollout), (s0_, d0, sbuf, dbuf) in zip(items, keep):
            want = src[rows] if per_rollout else src
            assert torch.equal(dst.view(torch.uint8), want.contiguous().view(torch.uint8)), (width, n_sc, per_rollout)
            assert torch.equal(sbuf, s0_)                               # the source is untouched
            assert torch.equal(dbuf[:64 + off], d0[:64 + off]) and torch.equal(dbuf[-64:], d0[-64:])  # guards
        # without a map every item is a plain copy
        for _, dst, _ in items:
            dst.zero_()
        ops.copy_rows(items, None, R)
        for src, dst, _ in items:
            assert torch.equal(dst.view(torch.uint8), src.view(torch.uint8))


def test_copy_rows_refuses_in_place_gather():
    x = torch.arange(64, dtype=torch.float32, device=DEV).view(8, 8)
    m = torch.tensor([1, 0, 3, 2, 1, 0, 3, 2], dtype=torch.int32, device=DEV)
    n0 = ops.LAUNCHES
    with pytest.raises(RuntimeError, match="unsupported"):
        ops.copy_rows([(x, x, True)], m, 4)
    assert ops.LAUNCHES == n0
    y = x.clone()
    ops.copy_rows([(x, x, True)], None, 4)                              # a plain in-place copy is harmless
    assert torch.equal(x, y)


# ---------------------------------------------------------------------------------------------- errors
def test_errors_launch_nothing():
    R, T = 4, 24
    eng, b, _ = _setup(0, R, T)
    with pytest.raises(RuntimeError):
        eng.snapshot()                                                  # nothing begun
    eng.prepare(b)
    with pytest.raises(RuntimeError):
        eng.snapshot()                                                  # prepared, not begun
    s0 = eng.begin(b)["t"]
    snap = eng.snapshot()
    _advance_to(eng, s0 + 2)
    torch.cuda.synchronize()
    live = {k: t.clone() for k, t, _ in eng._state_items()}
    n0 = ops.LAUNCHES
    for src in (torch.zeros(2, R), torch.zeros(2, R, dtype=torch.bool), torch.zeros(2, R + 1, dtype=torch.long),
                torch.zeros(R, dtype=torch.long), torch.full((2, R), R), torch.full((2, R), -1),
                torch.tensor([[0, 1, 2, 3], [0, 1, 2, 4]]), [[0, 0, 0, 0], [0, 0, 0, 0]]):
        with pytest.raises(ValueError):
            eng.restore(snap, src)
    with pytest.raises(TypeError):
        eng.restore(live)
    assert ops.LAUNCHES == n0 and eng._t == s0 + 2
    for k, t, _ in eng._state_items():
        assert torch.equal(t, live[k]), k
    eng.prepare(b)                                                      # the same batch again: a new generation
    with pytest.raises(RuntimeError):
        eng.restore(snap)
    eng.begin(b)
    with pytest.raises(RuntimeError):
        eng.restore(snap)
    snap2 = eng.snapshot()
    eng.begin({k: v[:1] for k, v in b.items()})                         # another shape: one scene
    assert eng._st["n_sc"] == 1
    with pytest.raises(RuntimeError):
        eng.restore(snap2)
    fresh = RolloutEngine(eng.model.P, eng.cfg, DEV, n_rollout=R, step_end=T)
    with pytest.raises(RuntimeError):
        fresh.restore(snap)                                             # no prepared batch
