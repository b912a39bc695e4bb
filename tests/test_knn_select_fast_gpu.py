"""The current KNN select kernels (early-exit bisection, the register-lean x-slab kernel of the agent -> map select)
against the previous ones (ops.knn_select(reference=True), TB_KNN_REFERENCE): idx, invalid flags, relative poses and
row states must be equal bit for bit, over the steps of a rollout and on adversarial inputs."""
import pytest
import torch

import tbpkg  # noqa: F401
from trafficbotsv1_5_b200 import config, ops, params, synth
from trafficbotsv1_5_b200.engine import RolloutEngine

from test_neighbour_stress_gpu import _grid_targets, _int_sources

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _both(src, sinv, tgt, tinv, K, lim, div=1, state=None, **kw):
    """Both kernel sets on the same inputs (each with its own copy of the row state); asserts equal outputs."""
    dv = lambda t: t.contiguous().to(DEV)  # noqa: E731
    outs = []
    for ref in (False, True):
        st = None if state is None else state.clone()
        outs.append(ops.knn_select(dv(src), dv(sinv), dv(tgt), dv(tinv), K, lim, tgt_div=div, row_state=st,
                                   reference=ref, **kw) + (st,))
    (i, m, r, s), (ri, rm, rr, rs) = outs
    assert torch.equal(i, ri), "idx"
    assert torch.equal(m, rm), "invalid"
    assert torch.equal(r.view(torch.int32), rr.view(torch.int32)), "rel"
    if state is not None:
        assert torch.equal(s.view(torch.int32), rs.view(torch.int32)), "row_state"
    return s


def _sorted_map(T, g, p_inv=0.15, lo=-40, hi=40):
    tgt, tinv = _grid_targets(1, T, g, p_inv=p_inv, lo=lo, hi=hi)
    order = torch.argsort(tgt[..., 0], dim=1, stable=True)
    pose = torch.gather(tgt, 1, order[..., None].expand(-1, -1, 3)).contiguous()
    return pose, torch.gather(tinv, 1, order).contiguous(), order.to(torch.int32).contiguous().to(DEV)


@pytest.mark.parametrize("T", [33, 64, 65, 120, 128, 129, 1024])
def test_small_and_full_scan_match_reference(T):
    """Exact distance ties at the K-th key, invalid sources, a scene with fewer valid targets than K, K up to T - 1,
    with and without a bracketing row state (agent -> TL)."""
    g = torch.Generator().manual_seed(T)
    B, S = 3, 40
    tgt, tinv = _grid_targets(B, T, g)
    tinv[1] = torch.rand(T, generator=g) < 0.9
    src, sinv = _int_sources(B, S, g)
    for K in sorted({k for k in (1, 8, 25, 32, 33, 64, T - 1) if k < T}):
        _both(src, sinv, tgt, tinv, K, 25.0)
        state = torch.full((B, S, 3), float("inf"), device=DEV)
        for step in range(4):
            state = _both(src, sinv, tgt, tinv, K, 25.0, state=state)
            src[..., :2] += torch.randint(-2, 3, (B, S, 2), generator=g).float()


@pytest.mark.parametrize("K", [25, 64])
def test_slab_kernel_matches_reference(K):
    """x-sorted static targets with a row state: the first call (state +inf), moving sources, a teleporting source,
    invalid sources and fewer valid targets than K in one scene."""
    g = torch.Generator().manual_seed(100 + K)
    B, S, T = 4, 70, 1024
    pose, inv, order = _sorted_map(T, g)
    pose2, inv2, order2 = _sorted_map(T, g)
    inv2[0, torch.randperm(T, generator=g)[: T - K // 2]] = True
    pose, inv = torch.cat([pose, pose2]), torch.cat([inv, inv2])
    order = torch.cat([order, order2])
    src, _ = _int_sources(B, S, g)
    state = torch.full((B, S, 3), float("inf"), device=DEV)
    for step in range(8):
        sinv = torch.rand(B, S, generator=g) < 0.1
        if step:
            src[..., :2] += torch.randint(-3, 4, (B, S, 2), generator=g).float()
        if step == 4:
            src[0, :5, :2] += 300.0  # teleport: the slab around the new position is empty
        state = _both(src, sinv, pose, inv, K, 20.0, div=2, state=state, index_map=order, sorted_by_x=True)


def test_slab_kernel_overflow_matches_reference():
    """More than 384 survivors in the slab (a stacked target cloud) and in the prune bound: the slab kernel's shared
    memory fallbacks (prune, then bisection over all keys) against the reference kernel's register paths."""
    g = torch.Generator().manual_seed(7)
    B, S, T = 2, 24, 1024
    pose, inv, order = _sorted_map(T, g, p_inv=0.05, lo=0, hi=3)
    pose[0, : T // 2, :2] = 1.0  # half the targets on one point
    pose[0] = pose[0][torch.argsort(pose[0, :, 0], stable=True)]
    src, sinv = _int_sources(B, S, g, lo=-2, hi=5)
    for K in (1, 32, 64, 65):
        state = torch.full((B, S, 3), float("inf"), device=DEV)
        for step in range(3):
            state = _both(src, sinv, pose, inv, K, 1e9, div=B, state=state, index_map=order, sorted_by_x=True)
            src[..., :2] += 1.0


def test_rollout_lists_match_reference():
    """24 steps of a config-3-shaped rollout (120 agent tokens, 1024 map tokens, 40 traffic-light tokens): each
    step's agent -> agent / map / TL lists, re-selected from the step's token poses by the reference kernels with
    their own row states, equal the engine's lists and row states."""
    cfg = config.default_model_cfg()
    R, n_steps = 4, 24
    eng = RolloutEngine(params.init_params(cfg, 0), cfg, DEV, precision=1, n_rollout=R, step_end=n_steps)
    eng.prepare(synth.make_scene_batch(n_sc=2, seed=11))
    st, mp, tl = eng._st, eng._static["mp"], eng._static["tl"]
    sz = eng.model.sz
    ref_state = ref_state_tl = None
    seen = []

    def record(s_, aux):
        nonlocal ref_state, ref_state_tl
        tp, ti = aux["tok_pose"], aux["tok_inv"]
        B, A = ti.shape
        if ref_state is None:
            ref_state = torch.full((B, A, 3), float("inf"), device=DEV)
            ref_state_tl = torch.full((B, A, 3), float("inf"), device=DEV)
        ks = aux["knn_self"]
        i, m, r = ops.knn_select(tp, ti, tp, ti, ks["idx"].shape[-1], sz["dl_ag"], reference=True)
        assert torch.equal(i, ks["idx"]) and torch.equal(m, ks["inv"]), f"step {s_}: agent -> agent"
        assert torch.equal(r.view(torch.int32), ks["rel"].view(torch.int32)), f"step {s_}: agent -> agent rel"
        Km = sz["k_ag2mp"]
        i, m, r = ops.knn_select(tp, ti, mp["mp_sorted_pose"], mp["mp_sorted_invalid"], Km, sz["dl_ag"],
                                 tgt_div=B // mp["mp_sorted_pose"].shape[0], index_map=mp["mp_sorted_index"],
                                 row_state=ref_state, sorted_by_x=True, reference=True)
        assert torch.equal(i, aux["cidx"][..., :Km]) and torch.equal(m, aux["cinv"][..., :Km]), f"step {s_}: map"
        assert torch.equal(r.view(torch.int32), aux["crel"][..., :Km, :].view(torch.int32)), f"step {s_}: map rel"
        assert torch.equal(ref_state.view(torch.int32), st["knn_state"].view(torch.int32)), f"step {s_}: map state"
        tlp, tli = tl["tl_token_pose"], tl["tl_token_invalid"]
        i, m, r = ops.knn_select(tp, ti, tlp, tli, sz["k_ag2tl"], sz["dl_ag"], tgt_div=B // tlp.shape[0],
                                 row_state=ref_state_tl, reference=True)
        assert torch.equal(i, aux["cidx"][..., Km:]) and torch.equal(m, aux["cinv"][..., Km:]), f"step {s_}: TL"
        assert torch.equal(r.view(torch.int32), aux["crel"][..., Km:, :].view(torch.int32)), f"step {s_}: TL rel"
        assert torch.equal(ref_state_tl.view(torch.int32), st["knn_state_tl"].view(torch.int32)), f"step {s_}: TL state"
        seen.append(s_)

    eng.run(record=record)
    assert len(seen) >= 20, seen
