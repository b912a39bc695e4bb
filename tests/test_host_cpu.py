"""Host-side logic that needs no GPU: weight re-association and layout permutations of the tensor-core mode."""
import torch

from oracle import tb_oracle as O
from trafficbotsv1_5_b200 import params
from trafficbotsv1_5_b200.model import H, fuse_attention, head_interleave_perm


def test_head_interleave_perm_layout():
    """tb_knarpe_attn flags bit 4: position 64*(h>>1) + 16*(c>>3) + 8*(h&1) + (c&7) holds channel c of head h — a
    permutation whose 32-byte pieces (16 halves) hold 8 channels of head 2i and 8 of head 2i+1."""
    perm = head_interleave_perm(128)
    assert sorted(perm.tolist()) == list(range(128))
    for h in range(4):
        for c in range(32):
            pos = 64 * (h >> 1) + 16 * (c >> 3) + 8 * (h & 1) + (c & 7)
            assert int(perm[pos]) == 32 * h + c
    pieces = perm.view(8, 16) // 32  # head of every channel, per 32-byte piece
    for i in range(8):
        assert pieces[i, :8].unique().tolist() == [2 * (i // 4)] and pieces[i, 8:].unique().tolist() == [2 * (i // 4) + 1]


def test_fused_attention_weights_reproduce_the_reference_formulation():
    """The re-associated projections (DESIGN.md 3: u = W_rk^T q, out-proj over [ov | z]) evaluated densely in torch
    equal the oracle's AttentionRPE (attention_rpe.py:137-190), including under the head-interleaved permutation of the
    q / k / v output features (a per-head permutation applied to q and k alike leaves q.k unchanged; v is un-permuted
    by the kernel's epilogue, modelled here by the inverse permutation)."""
    d, B, S, K = 128, 2, 5, 7
    g = torch.Generator().manual_seed(3)
    shapes = {"in_proj_weight": (3 * d, d), "in_proj_bias": (3 * d,), "out_proj_weight": (d, d), "out_proj_bias": (d,),
              "linear_rpe.weight": (2 * d, d), "linear_rpe.bias": (2 * d,)}
    sd = params.rand_like_state_dict(shapes, 5)
    P = {f"a.{k}": v for k, v in sd.items()}
    src, tgt = torch.randn(B, S, d, generator=g), torch.randn(B, S, K, d, generator=g)
    mask = torch.rand(B, S, K, generator=g) < 0.3
    mask[0, 0] = True
    rel = torch.cat([torch.randn(B, S, K, 2, generator=g) * 20, torch.randn(B, S, K, 1, generator=g)], -1)
    emb = O.pose_emb_xy_yaw(rel[..., :2], rel[..., 2], d)
    ref = O.attention_rpe(P, "a", src, tgt, mask, emb, H).double()

    f = {k: v.double() for k, v in fuse_attention(P, "a", d).items()}
    perm = head_interleave_perm(d)
    inv = torch.argsort(perm)
    for interleaved in (False, True):
        qu = src.double() @ f["w_in_q"].T + f["b_in_q"]
        kv = tgt.double() @ f["w_kv"].T + f["b_kv"]
        q, u, k, v = qu[..., :d], qu[..., d:].view(B, S, H, d), kv[..., :d], kv[..., d:]
        if interleaved:
            q, k, v = q[..., perm], k[..., perm], v[..., perm]
            head_of = (2 * (torch.arange(d) >> 6) + ((torch.arange(d) >> 3) & 1))
        else:
            head_of = torch.arange(d) // (d // H)
        sel = torch.nn.functional.one_hot(head_of, H).double()                       # [d, H]
        logit = torch.einsum("bsc,bskc,ch->bskh", q, k, sel) + torch.einsum("bshc,bskc->bskh", u, emb.double())
        logit = logit.masked_fill(mask[..., None], float("-inf"))
        a = torch.softmax(logit * 0.6931471805599453, dim=2)                         # q, u carry log2(e)
        a = torch.nan_to_num(a)
        ov = torch.einsum("bskh,bskc,ch->bsc", a, v, sel)
        if interleaved:
            ov = ov[..., inv]
        z = torch.einsum("bskh,bskc->bshc", a, emb.double()).reshape(B, S, H * d)
        out = torch.cat([ov, z], -1) @ f["w_out"].T + f["b_out"]
        out = out.masked_fill(mask.all(-1)[..., None], 0.0)
        assert float((out - ref).abs().max()) < 1e-5 * float(ref.abs().max()), interleaved


def test_knarpe_core_reference_composes_to_attention_rpe():
    """tests/_knarpe_ref.py (the float64 core the GPU stress tests compare against), composed with fuse_attention's
    packed projections, reproduces the oracle's AttentionRPE in float64: masked neighbours, an all-masked token, both
    model widths. The only difference is fuse_attention's fp32 rounding of the packed weights (2^-24 relative)."""
    import _knarpe_ref as KR
    for d, K in ((128, 9), (256, 5)):
        B, S = 2, 6
        g = torch.Generator().manual_seed(d + K)
        shapes = {"in_proj_weight": (3 * d, d), "in_proj_bias": (3 * d,), "out_proj_weight": (d, d),
                  "out_proj_bias": (d,), "linear_rpe.weight": (2 * d, d), "linear_rpe.bias": (2 * d,)}
        P = {f"a.{k}": v.double() for k, v in params.rand_like_state_dict(shapes, 7).items()}
        src, tgt = torch.randn(B, S, d, generator=g).double(), torch.randn(B, S, K, d, generator=g).double()
        mask = torch.rand(B, S, K, generator=g) < 0.3
        mask[1, 2] = True
        rel = torch.cat([torch.randn(B, S, K, 2, generator=g) * 30, torch.randn(B, S, K, 1, generator=g) * 2], -1).double()
        ref = O.attention_rpe(P, "a", src, tgt, mask, O.pose_emb_xy_yaw(rel[..., :2], rel[..., 2], d), H)
        out = KR.attention_from_core(fuse_attention(P, "a", d), src, tgt, mask, rel)
        assert out.dtype == torch.float64
        assert float((out - ref).abs().max()) < 1e-6 * float(ref.abs().max()), d
        assert float(out[1, 2].abs().max()) == 0.0


def test_rollout_buffer_layout_and_log_prob():
    """RolloutBuffer of the rollout-level drop-in (utils/buffer.py:103-146): joint-future flattening and the navigation
    log-probability average, on hand-made tensors (no GPU)."""
    from trafficbotsv1_5_b200.waymo_motion import RolloutBuffer, TeacherForcing, _check_teacher_forcing
    n_sc, R, A, T, n_tl = 2, 3, 4, 5, 2
    B = n_sc * R
    buf = RolloutBuffer(step_end=T, step_current=1)
    assert (buf.step_start, buf.step_end, buf.step_future_start) == (1, T, 1)
    lp0 = torch.arange(B * A, dtype=torch.float32).view(B, A)
    v0 = torch.ones(B, A, dtype=torch.bool)
    v0[0, 0] = False
    buf.add_navi_log_prob(lp0, v0)
    buf.add_navi_log_prob(lp0 * 3, torch.zeros(B, A, dtype=torch.bool))  # a later re-prediction nobody needed
    buf._finish()
    buf.pred_valid = torch.ones(B, A, T, dtype=torch.bool)
    buf.pred_pose = torch.zeros(B, A, T, 3)
    buf.pred_motion = torch.zeros(B, A, T, 3)
    buf.action_log_prob = torch.zeros(B, A, T)
    buf.mask_teacher_forcing = torch.zeros(B, A, T, dtype=torch.bool)
    buf.tl_state_nll = torch.zeros(B, n_tl, T)
    buf.tl_state_nll_invalid = torch.zeros(B, n_tl, T, dtype=torch.bool)
    buf.violation = {"collided": torch.zeros(B, A, T, dtype=torch.bool)}
    buf.flatten_joint_future(R)
    assert buf.pred_pose.shape == (n_sc, R, A, T, 3) and buf.navi_log_prob.shape == (n_sc, R, A, 2)
    assert buf.tl_state_nll.shape == (n_sc, R, n_tl, T) and buf.violation["collided"].shape == (n_sc, R, A, T)
    buf.compute_log_prob(torch.ones(B, A))
    exp = lp0.view(n_sc, R, A).clone() + 1
    exp[0, 0, 0] = 1.0  # no valid navigation sample: 0 (+ the latent term)
    assert torch.equal(buf.log_prob, exp)
    assert _check_teacher_forcing(TeacherForcing(step_spawn_agent=7, step_warm_start=9)) == (7, 9)


def test_3xtf32_weight_split_is_exact_and_cached():
    """ops._w3 (strict-parity projections on the tf32 tensor cores): [W | W | W - trunc_tf32(W)] where the truncation
    keeps sign, exponent and 10 mantissa bits. hi + lo must reproduce W bit for bit, lo must be below 2^-10 of |W|, and
    the split is rebuilt only when the weight tensor is modified in place; the 3-term sum x_hi W_hi + x_lo W_hi +
    x_hi W_lo (what one tf32 GEMM over [x | x_lo | x] . [W | W | W_lo] evaluates) drops only x_lo W_lo."""
    from trafficbotsv1_5_b200 import ops
    g = torch.Generator().manual_seed(0)
    w = torch.randn(40, 24, generator=g) * 10.0 ** torch.randint(-4, 4, (40, 1), generator=g)
    w3 = ops._w3(w)
    K = w.shape[1]
    assert w3.shape == (40, 3 * K) and torch.equal(w3[:, :K], w) and torch.equal(w3[:, K:2 * K], w)
    lo = w3[:, 2 * K:]
    hi = w - lo
    assert torch.equal(hi + lo, w)
    assert int((hi.view(torch.int32) & 0x1FFF).abs().max()) == 0          # 13 low mantissa bits cleared
    assert bool((lo.abs() <= w.abs() * 2.0 ** -10).all())
    assert ops._w3(w) is w3                                                # cached on the tensor object
    w.mul_(2.0)
    w3b = ops._w3(w)
    assert w3b is not w3 and torch.equal(w3b[:, :K], w)                    # in-place update -> rebuilt
    # the three-term product against float64: the dropped term is 2^-20 relative per product
    x = torch.randn(50, K, generator=g)
    trunc = lambda t: (t.view(torch.int32) & -8192).view(torch.float32)    # noqa: E731
    xh, wh = trunc(x), trunc(w)
    xl, wl = x - xh, w - wh
    three = xh.double() @ wh.double().T + xl.double() @ wh.double().T + xh.double() @ wl.double().T
    ref = x.double() @ w.double().T
    scale = (x.abs().double() @ w.abs().double().T)
    assert float(((three - ref).abs() / scale).max()) < 2.0 ** -19


def test_agent_compaction_keeps_every_valid_agent_in_order():
    """RolloutEngine._compact (host logic, no GPU): agent slots that are never valid in the ground truth are dropped,
    the kept slots are the valid ones in their original order (stable), the slot count is the largest per-scene valid
    count rounded up to 4 and at least k_ag2ag + 1, and every per-agent tensor of the batch is gathered consistently."""
    from trafficbotsv1_5_b200 import config, synth
    from trafficbotsv1_5_b200.engine import RolloutEngine
    cfg = config.default_model_cfg()
    batch = synth.make_scene_batch(n_sc=3, n_ag=64, n_mp=40, n_tl=6, seed=5)
    keep = torch.zeros(3, 64, dtype=torch.bool)
    keep[0, 3::2] = True        # 31 agents
    keep[1, :29] = True         # 29 agents
    keep[2, 10:45] = True       # 35 agents -> 36 slots
    batch["sc/ag_valid"] = batch["sc/ag_valid"] & keep[:, :, None]
    batch["sc/ag_valid"][:, :, 0] |= keep   # every kept agent is valid at least once
    eng = RolloutEngine.__new__(RolloutEngine)
    eng.compact_agents, eng.sz, eng.dev = True, config.derived_sizes(cfg), torch.device("cpu")
    out = eng._compact(batch)
    a_eff = out["sc/ag_valid"].shape[1]
    assert a_eff == 36 and eng._A_full == 64 and eng._perm.shape == (3, 36)
    ever = batch["sc/ag_valid"].any(-1)
    for sc in range(3):
        kept = eng._perm[sc].tolist()
        valid_ids = ever[sc].nonzero().flatten().tolist()
        assert kept[:len(valid_ids)] == valid_ids                        # valid first, original order
        assert not ever[sc][kept[len(valid_ids):]].any()                 # the rest is padding
        for k in ("sc/ag_valid", "sc/ag_pose", "sc/ag_motion", "sc/ag_attr"):
            if k in batch:
                assert torch.equal(out[k][sc], batch[k][sc][kept]), k
    assert out["agent/dest"].shape[1 if batch["agent/dest"].dim() == 2 else 2] == 36
    assert batch["sc/ag_valid"].shape[1] == 64                           # the caller's dict is untouched
    eng.compact_agents = False
    assert eng._compact(batch) is batch and eng._perm is None


def test_warm_start_invariant_step_count():
    """RolloutEngine._invariant_steps (host logic): the number of leading policy steps whose encoder inputs are the same
    for every rollout of a scene. With the test-time teacher forcing (warm start 10, spawn window 11) and gap-free
    tracks that is 11; an agent that is valid but NOT forced at time t (a track gap that closes after the spawn window,
    or a track that outlives the warm start) makes the state rollout-dependent from t on, so only steps 1 .. t qualify;
    fewer than 3 such steps switch the de-duplication off."""
    from trafficbotsv1_5_b200.engine import RolloutEngine, teacher_forcing_mask
    eng = RolloutEngine.__new__(RolloutEngine)
    eng.T = 90

    def s0(gt_valid, spawn=11, warm=10):
        tf = teacher_forcing_mask(gt_valid, spawn, warm)
        return eng._invariant_steps(dict(tf_mask=tf.to(torch.uint8), n_gt=gt_valid.shape[2]))

    gt = torch.ones(2, 5, 91, dtype=torch.bool)
    assert s0(gt) == 11                                   # times 0..10 forced; time 11 is the first free one
    late = gt.clone()
    late[1, 3, :7] = False                                # appears at t = 7 (inside the spawn window): forced there
    assert s0(late) == 11
    gap = gt.clone()
    gap[0, 2, 4] = False                                  # a gap at t = 4: the agent lives on under the policy there
    assert s0(gap) == 4                                   # (valid before, not forced) -> steps 1..4 only
    assert s0(gt, spawn=11, warm=3) == 4                  # warm start 3: times 0..3 forced, step 5 already differs
    assert s0(gt, spawn=0, warm=0) == 0                   # only time 0 forced: nothing worth batching
    short = torch.ones(1, 4, 8, dtype=torch.bool)
    assert s0(short) == 8                                 # bounded by the number of ground-truth steps
    eng.T = 6
    assert s0(gt) == 6                                    # and by the rollout length


def test_training_ring_index_matches_a_simulated_ring():
    """TrainStep._ring_index (host logic): the batched training pass rebuilds, for every policy step s, the history ring
    the step-by-step rollout would hold (slot = time % W, last W times). Simulate the ring write by write and compare."""
    from trafficbotsv1_5_b200.training import TrainStep
    ts = TrainStep.__new__(TrainStep)
    ts.dev = torch.device("cpu")
    for T, W in ((14, 11), (30, 11), (5, 11), (25, 4)):
        tidx, tmask = ts._ring_index(T, W)
        ring = [-1] * W                     # time stored in every slot, -1 = never written
        for s in range(1, T + 1):           # before step s the ring holds times 0 .. s-1 (the newest W of them)
            ring[(s - 1) % W] = s - 1
            for k in range(W):
                assert bool(tmask[s - 1, k]) == (ring[k] >= 0), (T, W, s, k)
                if ring[k] >= 0:
                    assert int(tidx[s - 1, k]) == ring[k], (T, W, s, k)
