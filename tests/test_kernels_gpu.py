"""GPU parity tests: every CUDA kernel (called through the C ABI via ops.*) against the CPU oracle and against
the golden vectors produced by the real reference. Tolerances are written next to each check."""
import pytest
import torch

import _knarpe_ref as KR
from oracle import tb_oracle as O
from trafficbotsv1_5_b200 import config, params

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from trafficbotsv1_5_b200 import ops
    from trafficbotsv1_5_b200.model import HotPathModel, fuse_attention, H

DEV = "cuda"


def close(a, b, rtol, atol, what):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    err = (a - b).abs()
    lim = atol + rtol * b.abs()
    bad = err > lim
    assert not bool(bad.any()), (f"{what}: {int(bad.sum())}/{bad.numel()} out of tol; max abs err "
                                 f"{float(err.max()):.3e} (ref max {float(b.abs().max()):.3e})")


def rel_l2(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


# ------------------------------------------------------------------------------------------------ knn select
def _knn_case(B, S, T, K, lim, seed, self_attn=False, div=1, p_inv=0.2):
    g = torch.Generator().manual_seed(seed)
    pose = torch.cat([(torch.rand(B, S, 2, generator=g) * 2 - 1) * 100, (torch.rand(B, S, 1, generator=g) * 2 - 1) * 3], -1)
    inv = torch.rand(B, S, generator=g) < p_inv
    if self_attn:
        return pose, inv, pose, inv
    Bt = B // div
    pose2 = torch.cat([(torch.rand(Bt, T, 2, generator=g) * 2 - 1) * 150, (torch.rand(Bt, T, 1, generator=g) * 2 - 1) * 3], -1)
    inv2 = torch.rand(Bt, T, generator=g) < p_inv
    return pose, inv, pose2, inv2


def _check_knn(pose, inv, pose2, inv2, K, lim, div=1):
    idx, knn_inv, rel = ops.knn_select(pose.to(DEV), inv.to(DEV), pose2.to(DEV), inv2.to(DEV), K, lim, tgt_div=div)
    idx, knn_inv, rel = idx.cpu().long(), knn_inv.cpu(), rel.cpu()
    p2, i2 = pose2.repeat_interleave(div, 0), inv2.repeat_interleave(div, 0)
    rel_pose, rel_dist = O.get_rel_pose(pose, inv, p2, i2)
    o_idx, o_inv, o_rel = O.knn_select(i2, rel_pose, rel_dist, K, lim)
    sd = torch.sort(rel_dist, -1)[0]
    # rows whose K-th / (K+1)-th distances are separated (tie-free) must match the oracle bit-exactly as SETS
    gap_ok = (sd[..., K] - sd[..., K - 1] > 1e-4 * sd[..., K - 1].clamp(min=1.0)) | ~torch.isfinite(sd[..., K - 1])
    d_sel = torch.gather(rel_dist, 2, idx)
    fin = torch.isfinite(d_sel)
    a = idx.masked_fill(~fin, -1).sort(-1)[0]
    b = o_idx.masked_fill(~torch.isfinite(torch.gather(rel_dist, 2, o_idx)), -1).sort(-1)[0]
    assert torch.equal(a[gap_ok], b[gap_ok]), "KNN index sets differ on tie-free rows"
    assert int(gap_ok.sum()) > 0.9 * gap_ok.numel()
    # selected indices are distinct and in range; emitted in ascending index order
    assert bool((idx[..., 1:] > idx[..., :-1]).all())
    assert int(idx.min()) >= 0 and int(idx.max()) < pose2.shape[1]
    # invalid flag and relative pose of every selected neighbour (1e-4 m / 1e-6 rad abs: fp32 rotation rounding)
    exp_inv = torch.gather(i2[:, None].expand(-1, pose.shape[1], -1), 2, idx) | (d_sel > lim)
    near = (d_sel - lim).abs() < 1e-3
    assert torch.equal(knn_inv | near, exp_inv | near)
    exp_rel = torch.gather(rel_pose, 2, idx[..., None].expand(-1, -1, -1, 3))
    close(rel[fin][:, :2], exp_rel[fin][:, :2], 0, 1e-4, "rel xy")
    close(rel[..., 2], exp_rel[..., 2], 0, 1e-6, "rel yaw")


@pytest.mark.parametrize("B,S,T,K,lim,self_attn,div", [
    (2, 24, 50, 12, 60.0, False, 1), (3, 40, 40, 24, 250.0, True, 1), (4, 128, 1024, 64, 500.0, False, 2),
    (2, 128, 128, 25, 500.0, True, 1), (6, 128, 40, 25, 500.0, False, 3), (1, 7, 33, 32, 1e9, False, 1),
    (1, 70, 2048, 100, 80.0, False, 1), (2, 5, 300, 1, 100.0, False, 1)])
def test_knn_select_vs_oracle(B, S, T, K, lim, self_attn, div):
    _check_knn(*_knn_case(B, S, T, K, lim, 100 + T + K, self_attn, div), K, lim, div)


def test_knn_select_all_invalid_and_errors():
    pose, inv, pose2, inv2 = _knn_case(1, 8, 64, 10, 100.0, 5)
    inv[:] = True
    idx, kinv, _ = ops.knn_select(pose.to(DEV), inv.to(DEV), pose2.to(DEV), inv2.to(DEV), 10, 100.0)
    assert bool(kinv.all())
    with pytest.raises(RuntimeError):  # reference assert 0 < K < T (utils/rpe.py:79)
        ops.knn_select(pose.to(DEV), inv.to(DEV), pose2.to(DEV), inv2.to(DEV), 64, 100.0)


@pytest.mark.parametrize("name", ["knn_small", "knn_self_", "knn_big"])
def test_knn_select_golden(golden_ops, name):
    g = golden_ops[name]
    p2 = g["pose"] if g["pose2"] is None else g["pose2"]
    i2 = g["inv"] if g["inv2"] is None else g["inv2"]
    idx, kinv, rel = ops.knn_select(g["pose"].to(DEV), g["inv"].to(DEV), p2.to(DEV), i2.to(DEV), g["K"], g["lim"])
    fin = torch.isfinite(g["dist"])
    # golden rows are sorted by distance, ours by index: compare as sets (inf fillers free)
    a = idx.cpu().long()
    rel_pose, rel_dist = O.get_rel_pose(g["pose"], g["inv"], g["pose2"], g["inv2"])
    mine_fin = torch.isfinite(torch.gather(rel_dist, 2, a))
    assert torch.equal(a.masked_fill(~mine_fin, -1).sort(-1)[0], g["idx"].masked_fill(~fin, -1).sort(-1)[0])
    assert int(kinv.sum()) == int(g["knn_inv"].sum())


# ------------------------------------------------------------------------------------------------ small ops
@pytest.mark.parametrize("M,N,K,flags", [(300, 128, 128, "b"), (1000, 896, 128, "b"), (77, 5, 128, "b"),
                                         (513, 121, 31, "br"), (200, 121, 121, "b"), (129, 64, 128, "brm"),
                                         (640, 128, 640, "bpr+"), (50, 2, 128, ""), (4097, 512, 128, "br"),
                                         (333, 128, 512, "b+q")])
def test_linear_f32(M, N, K, flags):
    g = torch.Generator().manual_seed(M + N)
    x, w, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / K ** 0.5, torch.randn(N, generator=g)
    res = torch.randn(M, N, generator=g)
    mp, mq = torch.rand(M, generator=g) < 0.3, torch.rand(M, generator=g) < 0.3
    y = torch.nn.functional.linear(x.double(), w.double(), b.double() if "b" in flags else None)
    kw = {}
    if "r" in flags:
        y = y.relu(); kw["relu"] = True
    if "p" in flags or "m" in flags:
        y = y.masked_fill(mp[:, None], 0); kw["mask_pre"] = mp.to(DEV)
    if "+" in flags:
        y = y + res.double(); kw["res"] = res.to(DEV)
    if "q" in flags:
        y = y.masked_fill(mq[:, None], 0); kw["mask_post"] = mq.to(DEV)
    out = ops.linear(x.to(DEV), w.to(DEV), b.to(DEV) if "b" in flags else None, **kw)
    close(out, y.float(), 1e-5, 1e-5, f"linear {M}x{N}x{K} {flags}")  # fp32 FFMA vs float64: 1e-5


def test_linear_strided_views():
    g = torch.Generator().manual_seed(3)
    x = torch.randn(100, 384, generator=g).to(DEV)
    w = (torch.randn(128, 128, generator=g) / 11).to(DEV)
    out = torch.zeros(100, 384, device=DEV)
    ops.linear(x[:, 128:256], w, None, out=out[:, 256:])
    close(out[:, 256:], x[:, 128:256] @ w.T, 1e-5, 1e-5, "strided linear")
    assert float(out[:, :256].abs().max()) == 0.0


@pytest.mark.parametrize("D", [128, 256])
def test_layernorm(D):
    g = torch.Generator().manual_seed(D)
    x, w, b = torch.randn(333, D, generator=g) * 3 + 1, torch.randn(D, generator=g), torch.randn(D, generator=g)
    y = torch.nn.functional.layer_norm(x, (D,), w, b, 1e-5)
    close(ops.layernorm(x.to(DEV), w.to(DEV), b.to(DEV)), y, 1e-5, 1e-5, "layernorm")
    close(ops.layernorm(x.to(DEV), w.to(DEV), b.to(DEV), relu=True), y.relu(), 1e-5, 1e-5, "layernorm + relu")
    yh = ops.layernorm(x.to(DEV), w.to(DEV), b.to(DEV), out_dtype=torch.float16)
    assert yh.dtype == torch.float16 and torch.equal(yh.cpu(), ops.layernorm(x.to(DEV), w.to(DEV), b.to(DEV)).cpu().half())


@pytest.mark.parametrize("pe", [64, 128, 256])
def test_pose_emb(golden_ops, pe):
    g = golden_ops[f"pe_{pe}"]
    pose = torch.cat([g["xy"], g["yaw"]], -1).reshape(-1, 3)
    out = ops.pose_emb(pose.to(DEV), ops.pe_freq_xy(pe, 1e3, DEV), pe)
    # SFU sin/cos after exact 2-term range reduction: 2e-6 abs (documented 2^-21.4 on [-pi,pi])
    close(out, g["emb"].reshape(-1, pe), 0, 2e-6, f"pose_emb {pe}")


def test_pose_emb_frame():
    g = torch.Generator().manual_seed(9)
    pose = torch.cat([(torch.rand(50, 2, generator=g) * 2 - 1) * 200, (torch.rand(50, 1, generator=g) * 2 - 1) * 3], -1)
    frame = torch.cat([(torch.rand(50, 2, generator=g) * 2 - 1) * 200, (torch.rand(50, 1, generator=g) * 2 - 1) * 3], -1)
    xy = O.to_local_xy(pose[:, None, :2], frame[:, None, :2], frame[:, 2]).squeeze(1)
    ref = O.pose_emb_xy_yaw(xy, pose[:, 2] - frame[:, 2], 128)
    out = ops.pose_emb(pose.to(DEV), ops.pe_freq_xy(128, 1e3, DEV), 128, frame=frame.to(DEV))
    close(out, ref, 0, 1e-4, "pose_emb in frame")  # 1e-4: fp32 rounding of the rotated x,y times f_0 = 1 rad/m


def test_pointnet(golden_ops):
    cfg = config.default_model_cfg()
    P = params.init_params(cfg, 3)
    g = torch.Generator().manual_seed(4)
    B, N, Lg, d = 3, 17, 11, 128
    x = torch.randn(B, N, Lg, d, generator=g)
    inv = torch.rand(B, N, Lg, generator=g) < 0.4
    inv[0, 0] = True
    ref = O.pointnet(P, "ag_encoder.temp_encoder", x, inv)
    m = HotPathModel(P, cfg, config.derived_sizes(cfg), DEV)
    out = m.pointnet(x.reshape(-1, d).to(DEV), inv.reshape(-1).to(DEV), B * N, Lg, "ag_encoder.temp_encoder")
    close(out, ref.reshape(-1, d), 1e-5, 1e-5, "pointnet")
    assert float(out[0].abs().max()) == 0.0


# ------------------------------------------------------------------------------------------------ KNARPE attention
def _run_attention(sd, src, tgt, mask, rel, use_emb=False, half_kv=False, half_qu=False, **flags):
    """AttentionRPE semantics with an arbitrary pre-gathered tgt [B,S,K,d]: table = tgt flattened, idx = s*K+k."""
    B, S, K, d = tgt.shape
    P = {f"a.{k}": v for k, v in sd.items()}
    f = {k: v.to(DEV) for k, v in fuse_attention(P, "a", d).items()}
    if flags.get("interleaved"):  # tb_knarpe_attn flags bit 4: q / k / v output features stored head-interleaved
        from trafficbotsv1_5_b200.model import head_interleave_perm
        perm = head_interleave_perm(d).to(DEV)
        rq = torch.arange(d + H * d, device=DEV)
        rq[:d] = perm
        rkv = torch.cat([perm, d + perm])
        f = dict(f, w_in_q=f["w_in_q"][rq].contiguous(), b_in_q=f["b_in_q"][rq].contiguous(),
                 w_kv=f["w_kv"][rkv].contiguous(), b_kv=f["b_kv"][rkv].contiguous())
    if half_qu:  # fp16 [q|u] rows straight from the projection's epilogue (tensor-core mode)
        proj = torch.empty(B * S, d + H * d, dtype=torch.float16, device=DEV)
        ops.linear(src.reshape(B * S, d).to(DEV), f["w_in_q"], f["b_in_q"], precision=1, out_h=proj, col_h=0)
    else:
        proj = ops.linear(src.reshape(B * S, d).to(DEV), f["w_in_q"], f["b_in_q"])
    if half_kv:  # tensor-core mode: the projection writes the fp16 table (tf32 MMA), the attention runs on mma.sync
        kv = torch.empty(B * S * K, 2 * d, dtype=torch.float16, device=DEV)
        ops.linear(tgt.reshape(B * S * K, d).to(DEV), f["w_kv"], f["b_kv"], precision=1, out_h=kv, col_h=0)
    else:
        kv = ops.linear(tgt.reshape(B * S * K, d).to(DEV), f["w_kv"], f["b_kv"])
    idx = torch.arange(S * K, dtype=torch.int32, device=DEV).view(1, S, K).expand(B, -1, -1).contiguous()
    freq = ops.pe_freq_xy(d, 1e3, DEV)
    emb = O.pose_emb_xy_yaw(rel[..., :2], rel[..., 2], d).to(DEV).contiguous() if use_emb else None
    o, nv = ops.knarpe_attn(proj[:, :d], proj[:, d:], kv, S * K, 1, K, idx, mask.to(DEV).contiguous(),
                            None if use_emb else rel.to(DEV).contiguous(), freq, B, S, d, H, emb=emb, **flags)
    if o.dtype == torch.float16:  # fp16 [ov|z] rows feed a kind::f16 out-projection
        out = ops.linear(o, f["w_out"].half().contiguous(), f["b_out"], mask_pre=nv, precision=2)
    else:
        out = ops.linear(o, f["w_out"], f["b_out"], mask_pre=nv)
    return out.view(B, S, d), nv.view(B, S)


def test_attention_d256_16bit_golden(golden_ops):
    """BASELINE config 2's model size (d_model 256, 4 heads of 64, K = 36) in the 16-bit mode: fp16 [q|u] rows, fp16
    K|V table, the SIMT core on fp16 tables (tb_knarpe_attn flags bit 1 with D = 256), fp16 [ov|z] rows, against the
    real reference's fp32 output. Stated 16-bit tolerance: 4e-3 of the output scale, 1.5e-3 in L2 (10-bit-mantissa
    operands; bf16 would be 4x coarser), all-masked rows exactly zero. Also through the drop-in module."""
    from trafficbotsv1_5_b200 import reference_api as R
    g = golden_ops["attn_d256"]
    sd = params.rand_like_state_dict(g["sd_shapes"], g["sd_seed"])
    out, nv = _run_attention(sd, g["src"], g["tgt"], g["mask"], g["rel"], half_kv=True, half_qu=True, fast_trig=True,
                             out_dtype=torch.float16)
    scale = float(g["out"].abs().max())
    print("d256 16-bit: max abs / scale", float((out.cpu() - g["out"]).abs().max()) / scale, "rel_l2", rel_l2(out, g["out"]))
    close(out, g["out"], 4e-3, 4e-3 * scale, "attn_d256 16-bit")
    assert rel_l2(out, g["out"]) < 1.5e-3
    assert bool(nv[0, 0]) and float(out[0, 0].abs().max()) == 0.0
    att = R.AttentionRPE(256, 4, dropout_p=0.1, bias=True, d_rpe=256, precision=1).eval()
    att.load_state_dict(sd)
    att = att.to(DEV)
    o2, _ = att(g["src"].to(DEV), g["tgt"].to(DEV), tgt_padding_mask=g["mask"].to(DEV), rpe=g["rel"].to(DEV))
    close(o2, g["out"], 4e-3, 4e-3 * scale, "drop-in AttentionRPE d256 16-bit")
    att.precision = 0
    att._tb_ver = None
    o3, _ = att(g["src"].to(DEV), g["tgt"].to(DEV), tgt_padding_mask=g["mask"].to(DEV), rpe=g["rel"].to(DEV))
    close(o3, g["out"], 1e-4, 1e-4 * scale, "drop-in AttentionRPE d256 fp32")


@pytest.mark.parametrize("name", ["attn_d128", "attn_d256"])
@pytest.mark.parametrize("use_emb", [False, True])
def test_attention_golden(golden_ops, name, use_emb):
    g = golden_ops[name]
    sd = params.rand_like_state_dict(g["sd_shapes"], g["sd_seed"])
    out, nv = _run_attention(sd, g["src"], g["tgt"], g["mask"], g["rel"], use_emb)
    # north star: attention outputs within 1e-4 relative in fp32 (relative to the output scale)
    scale = float(g["out"].abs().max())
    close(out, g["out"], 1e-4, 1e-4 * scale, f"{name} emb={use_emb}")
    assert rel_l2(out, g["out"]) < 2e-5
    assert bool(nv[0, 0]) and float(out[0, 0].abs().max()) == 0.0  # all-masked row -> exact zero


@pytest.mark.parametrize("d,B,S,K", [(128, 2, 130, 89), (128, 1, 64, 25), (256, 1, 40, 36), (128, 3, 33, 1)])
def test_attention_vs_oracle_and_properties(d, B, S, K):
    g = torch.Generator().manual_seed(d + K)
    shapes = {"in_proj_weight": (3 * d, d), "in_proj_bias": (3 * d,), "out_proj_weight": (d, d), "out_proj_bias": (d,),
              "linear_rpe.weight": (2 * d, d), "linear_rpe.bias": (2 * d,)}
    sd = params.rand_like_state_dict(shapes, 21)
    src, tgt = torch.randn(B, S, d, generator=g), torch.randn(B, S, K, d, generator=g)
    mask = torch.rand(B, S, K, generator=g) < 0.3
    mask[0, 1] = True
    rel = torch.cat([(torch.rand(B, S, K, 2, generator=g) * 2 - 1) * 300, (torch.rand(B, S, K, 1, generator=g) * 2 - 1) * 7], -1)
    P = {f"a.{k}": v for k, v in sd.items()}
    ref = O.attention_rpe(P, "a", src, tgt, mask, O.pose_emb_xy_yaw(rel[..., :2], rel[..., 2], d), H)
    out, _ = _run_attention(sd, src, tgt, mask, rel)
    scale = float(ref.abs().max())
    close(out, ref, 1e-4, 1e-4 * scale, "attention vs oracle")
    assert float(out[0, 1].abs().max()) == 0.0
    # permutation invariance over the neighbour order (fp summation order only): 1e-5 relative
    perm = torch.randperm(K, generator=g)
    out_p, _ = _run_attention(sd, src, tgt[:, :, perm], mask[:, :, perm], rel[:, :, perm])
    close(out_p, out, 1e-5, 1e-5 * scale, "permutation invariance")


@pytest.mark.parametrize("B,S,K,p_mask", [(2, 130, 89, 0.3), (1, 64, 25, 0.0), (3, 33, 1, 0.0), (1, 50, 64, 0.9),
                                          (2, 40, 112, 0.5)])
def test_attention_tensor_core(B, S, K, p_mask):
    """flags bit 1: fp16 K|V tables (written by the tf32 projection) and all four contractions on mma.sync with fp16
    k / v / e and split-fp16 q / u / p. Error budget = 2^-11 relative rounding of k, v, e + the tf32 table projection:
    3e-3 of the output scale, 1e-3 in L2 (same order as a tf32 projection, see test_linear_tensor_core)."""
    d = 128
    g = torch.Generator().manual_seed(K + S)
    shapes = {"in_proj_weight": (3 * d, d), "in_proj_bias": (3 * d,), "out_proj_weight": (d, d), "out_proj_bias": (d,),
              "linear_rpe.weight": (2 * d, d), "linear_rpe.bias": (2 * d,)}
    sd = params.rand_like_state_dict(shapes, 22)
    src, tgt = torch.randn(B, S, d, generator=g), torch.randn(B, S, K, d, generator=g)
    mask = torch.rand(B, S, K, generator=g) < p_mask
    mask[0, 1] = True
    rel = torch.cat([(torch.rand(B, S, K, 2, generator=g) * 2 - 1) * 300, (torch.rand(B, S, K, 1, generator=g) * 2 - 1) * 3.2], -1)
    P = {f"a.{k}": v for k, v in sd.items()}
    ref = O.attention_rpe(P, "a", src, tgt, mask, O.pose_emb_xy_yaw(rel[..., :2], rel[..., 2], d), H)
    out, nv = _run_attention(sd, src, tgt, mask, rel, half_kv=True, fast_trig=True)
    scale = float(ref.abs().max())
    print("tensor-core attention: max abs / scale", float((out.cpu() - ref).abs().max()) / scale, "rel_l2", rel_l2(out, ref))
    close(out, ref, 3e-3, 3e-3 * scale, "tensor-core attention vs oracle")
    assert rel_l2(out, ref) < 1e-3
    assert bool(nv[0, 1]) and float(out[0, 1].abs().max()) == 0.0
    assert torch.equal(nv.cpu(), mask.all(-1))


def _block_P(g):
    return {f"b.{k}": v for k, v in params.rand_like_state_dict(g["sd_shapes"], g["sd_seed"]).items()}


@pytest.mark.parametrize("mode", ["enc_self_attn", "dec_cross_attn"])
def test_transformer_block_golden(golden_ops, mode):
    g = golden_ops[f"block_{mode}"]
    P = _block_P(g)
    cfg = config.default_model_cfg()
    full = params.init_params(cfg, 0)
    full.update(P)
    m = HotPathModel(full, cfg, config.derived_sizes(cfg), DEV)
    B, S, d = g["src"].shape
    src = g["src"].reshape(B * S, d).to(DEV)
    inv = g["src_inv"].reshape(-1).to(DEV)
    knn_self = dict(idx=g["idx"].to(DEV, torch.int32).contiguous(), inv=g["m1"].to(DEV).contiguous(),
                    rel=g["rel1"].to(DEV).contiguous())
    for i in range(g["n_layer"]):
        p = f"b.layers.{i}"
        cross = None
        if mode == "dec_cross_attn":
            T2 = g["tgt_tab"].shape[1]
            kv = m.kv_table(g["tgt_tab"].reshape(-1, d).to(DEV), p, "norm_tgt")
            cross = dict(kv0=kv, T0=T2, div0=1, K0=g["idx2"].shape[-1], idx=g["idx2"].to(DEV, torch.int32).contiguous(),
                         inv=g["m2"].to(DEV).contiguous(), rel=g["rel2"].to(DEV).contiguous())
        src = m.tf_layer(p, mode, src, inv, B, S, knn_self, cross)
    scale = float(g["out"].abs().max())
    close(src.view(B, S, d), g["out"], 1e-4, 1e-4 * scale, f"block {mode}")
    assert rel_l2(src.view(B, S, d), g["out"]) < 2e-5


# ------------------------------------------------------------------------------------------------ tcgen05 projections
@pytest.mark.parametrize("M,N,K,flags", [(300, 128, 128, "b"), (1000, 896, 128, "b"), (4097, 512, 128, "br"),
                                         (640, 128, 640, "bpr+"), (129, 64, 128, "brm"), (720, 64, 20, "br"),
                                         (333, 128, 512, "b+q"), (77, 40, 16, "b"), (65536, 640, 128, "b"),
                                         (50, 384, 128, "br")])
def test_linear_tensor_core(M, N, K, flags):
    """precision=1: tcgen05 kind::tf32 (10-bit mantissa operands, fp32 accumulate). Stated tolerance: 2e-3 of the
    output scale (rms) per element — vs 1e-5 for the fp32 FFMA path."""
    g = torch.Generator().manual_seed(M + N)
    x, w, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / K ** 0.5, torch.randn(N, generator=g)
    res = torch.randn(M, N, generator=g)
    mp, mq = torch.rand(M, generator=g) < 0.3, torch.rand(M, generator=g) < 0.3
    y = torch.nn.functional.linear(x.double(), w.double(), b.double() if "b" in flags else None)
    kw = {}
    if "r" in flags:
        y = y.relu(); kw["relu"] = True
    if "p" in flags or "m" in flags:
        y = y.masked_fill(mp[:, None], 0); kw["mask_pre"] = mp.to(DEV)
    if "+" in flags:
        y = y + res.double(); kw["res"] = res.to(DEV)
    if "q" in flags:
        y = y.masked_fill(mq[:, None], 0); kw["mask_post"] = mq.to(DEV)
    out = ops.linear(x.to(DEV), w.to(DEV), b.to(DEV) if "b" in flags else None, precision=1, **kw)
    torch.cuda.synchronize()
    err = (out.cpu().double() - y).abs()
    scale = float(y.std())
    print(f"tf32 linear {M}x{N}x{K} {flags}: max err {float(err.max()):.3e}, rms err {float(err.pow(2).mean().sqrt()):.3e}, "
          f"out rms {scale:.3e}")
    assert float(err.max()) < 4e-3 * max(scale, 1.0), "tf32 projection out of tolerance"
    assert float(err.pow(2).mean().sqrt()) < 1e-3 * max(scale, 1.0)


@pytest.mark.parametrize("M,N,K,flags", [(1024, 128, 128, "b"), (4097, 512, 128, "br"), (2000, 128, 640, "bpr+"),
                                         (65536, 640, 128, "b"), (3000, 64, 20, "br"), (1500, 384, 256, "b+q"),
                                         (500, 128, 128, "b"), (2048, 128, 18, "b")])
def test_linear_3xtf32(M, N, K, flags):
    """precision=3: the strict-parity projections on the tensor cores. The activation rows are split into
    [x | x - trunc(x) | x] (tb_tf32_split3), the weights into [W | W | W - trunc(W)], and one kind::tf32 GEMM over 3K
    sums x_hi W_hi + x_lo W_hi + x_hi W_lo. The operand error is 2^-21 per product; what remains is the tensor core's
    round-toward-zero fp32 accumulate (one truncation per K=8 instruction, 3K/8 of them), a bias that grows linearly
    with K: measured 1.2e-5 (K=128) .. 4.4e-5 (K=640) of the output scale against 2.5e-6 .. 4.7e-6 for the FFMA kernel.
    Stated tolerance: (1e-5 + 6e-8 * 3K/8 * 4) of the output scale per element; shapes the split cannot take
    (M < 1024, K % 4) must fall back to the FFMA kernel."""
    g = torch.Generator().manual_seed(M + N + 1)
    x, w, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / K ** 0.5, torch.randn(N, generator=g)
    res = torch.randn(M, N, generator=g)
    mp, mq = torch.rand(M, generator=g) < 0.3, torch.rand(M, generator=g) < 0.3
    y = torch.nn.functional.linear(x.double(), w.double(), b.double() if "b" in flags else None)
    kw = {}
    if "r" in flags:
        y = y.relu(); kw["relu"] = True
    if "p" in flags:
        y = y.masked_fill(mp[:, None], 0); kw["mask_pre"] = mp.to(DEV)
    if "+" in flags:
        y = y + res.double(); kw["res"] = res.to(DEV)
    if "q" in flags:
        y = y.masked_fill(mq[:, None], 0); kw["mask_post"] = mq.to(DEV)
    wd = w.to(DEV)
    out = ops.linear(x.to(DEV), wd, b.to(DEV) if "b" in flags else None, precision=3, **kw)
    out0 = ops.linear(x.to(DEV), wd, b.to(DEV) if "b" in flags else None, precision=0, **kw)
    torch.cuda.synchronize()
    err = (out.cpu().double() - y).abs()
    err0 = (out0.cpu().double() - y).abs()
    scale = max(float(y.std()), 1.0)
    print(f"3xtf32 linear {M}x{N}x{K} {flags}: max err {float(err.max()):.3e} (FFMA kernel {float(err0.max()):.3e}), "
          f"out rms {scale:.3e}")
    assert float(err.max()) < (1e-5 + 6e-8 * (3 * K / 8) * 4) * scale, "3xTF32 projection out of tolerance"
    if M < 1024 or K % 4:
        assert torch.equal(out, out0), "shapes outside the split must run the FFMA kernel"
    else:
        assert hasattr(wd, "_tb_w3") and wd._tb_w3[1].shape == (N, 3 * K)


def test_tf32_split3_bits():
    """tb_tf32_split3: column blocks 0 and 2 are the input bit-for-bit, block 1 is x minus its 10-mantissa-bit
    truncation (exactly representable, so the comparison is bit-exact); misaligned K is refused."""
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(1031, 132, generator=g) * 10.0 ** torch.randint(-3, 4, (1031, 1), generator=g)).to(DEV)
    xs = x[:, 4:]  # strided view (ld 132, K 128)
    out = ops.tf32_split3(xs)
    hi = (xs.contiguous().view(torch.int32) & -8192).view(torch.float32)
    assert torch.equal(out[:, :128], xs) and torch.equal(out[:, 256:], xs)
    assert torch.equal(out[:, 128:256], xs - hi)
    with pytest.raises(RuntimeError):
        ops.tf32_split3(x[:, :130])


def test_linear_tensor_core_strided():
    g = torch.Generator().manual_seed(3)
    x = torch.randn(1000, 384, generator=g).to(DEV)
    w = (torch.randn(128, 128, generator=g) / 11).to(DEV)
    out = torch.zeros(1000, 384, device=DEV)
    ops.linear(x[:, 128:256], w, None, out=out[:, 256:], precision=1)
    ref = x[:, 128:256].double() @ w.double().T
    assert float((out[:, 256:].double() - ref).abs().max()) < 4e-3
    assert float(out[:, :256].abs().max()) == 0.0


# ------------------------------------------------------------------------------------------------ drop-in module API
def test_dropin_modules_golden(golden_ops):
    """reference-style calls (state_dict loading, materialised PoseEmb rpe, gathered tgt) through the drop-in classes."""
    from trafficbotsv1_5_b200 import reference_api as R
    g = golden_ops["attn_d128"]
    att = R.AttentionRPE(128, 4, dropout_p=0.1, bias=True, d_rpe=128).eval()
    att.load_state_dict(params.rand_like_state_dict(g["sd_shapes"], g["sd_seed"]))
    att = att.to(DEV)
    pe = R.PoseEmb("pe_xy_yaw", pe_dim=128, theta_xy=1e3).to(DEV)
    rel = g["rel"].to(DEV)
    out, w = att(g["src"].to(DEV), g["tgt"].to(DEV), tgt_padding_mask=g["mask"].to(DEV),
                 rpe=pe(rel[..., :2], rel[..., 2:3]))
    assert w is None
    close(out, g["out"], 1e-4, 1e-4 * float(g["out"].abs().max()), "drop-in AttentionRPE")
    with pytest.raises(NotImplementedError):
        att(g["src"].to(DEV), g["tgt"].to(DEV), rpe=None)
    for mode in ("enc_self_attn", "dec_cross_attn"):
        b = golden_ops[f"block_{mode}"]
        blk = R.TransformerBlockRPE(d_model=128, n_head=4, k_feedforward=4, dropout_p=0.1, bias=True, activation="relu",
                                    out_layernorm=False, apply_q_rpe=False, n_layer=b["n_layer"], mode=mode, d_rpe=128)
        missing, unexpected = blk.load_state_dict(params.rand_like_state_dict(b["sd_shapes"], b["sd_seed"]), strict=True)
        blk = blk.eval().to(DEV)
        e = lambda r: pe(r.to(DEV)[..., :2], r.to(DEV)[..., 2:3])  # noqa: E731
        if mode == "enc_self_attn":
            out, _ = blk(src=b["src"].to(DEV), src_padding_mask=b["src_inv"].to(DEV), tgt=b["idx"].to(DEV),
                         tgt_padding_mask=b["m1"].to(DEV), rpe=e(b["rel1"]))
        else:
            tgt = b["tgt_tab"][torch.arange(b["src"].shape[0])[:, None, None], b["idx2"]].to(DEV)
            out, _ = blk(src=b["src"].to(DEV), src_padding_mask=b["src_inv"].to(DEV), tgt=tgt,
                         tgt_padding_mask=b["m2"].to(DEV), rpe=e(b["rel2"]), decoder_tgt=b["idx"].to(DEV),
                         decoder_tgt_padding_mask=b["m1"].to(DEV), decoder_rpe=e(b["rel1"]))
        close(out, b["out"], 1e-4, 1e-4 * float(b["out"].abs().max()), f"drop-in block {mode}")
    # utils.rpe mirror
    k = golden_ops["knn_small"]
    rp, rd = R.get_rel_pose(k["pose"].to(DEV), k["inv"].to(DEV), k["pose2"].to(DEV), k["inv2"].to(DEV))
    idx, kinv, rpe3 = R.get_tgt_knn_idx(k["inv2"].to(DEV), rp, rd, k["K"], k["lim"])
    assert idx.dtype == torch.int64 and rpe3.shape[-1] == 3
    with pytest.raises(AssertionError):
        R.get_tgt_knn_idx(k["inv2"].to(DEV), rp, rd, k["pose2"].shape[1], k["lim"])


@pytest.mark.parametrize("prec", [0, 1])
@pytest.mark.parametrize("M,N,K,g", [(1100, 64, 64, 11), (257, 128, 128, 20), (330, 40, 64, 11)])
def test_linear_grouped_bias(M, N, K, g, prec):
    """bias_group: one bias row per group of g consecutive rows (de-duplicated PointNet, polyline_encoder.py:52)."""
    gen = torch.Generator().manual_seed(M)
    x, w = torch.randn(M, K, generator=gen), torch.randn(N, K, generator=gen) / K ** 0.5
    gb = torch.randn((M + g - 1) // g, N, generator=gen)
    ref = (x.double() @ w.double().T + gb.double().repeat_interleave(g, 0)[:M]).relu()
    out = ops.linear(x.to(DEV), w.to(DEV), gb.to(DEV), relu=True, bias_group=g, precision=prec)
    tol = 1e-5 if prec == 0 else 4e-3
    close(out, ref.float(), tol, tol, f"grouped bias prec={prec}")


@pytest.mark.parametrize("M,N,K", [(1000, 6, 384), (640, 5, 128), (300, 2, 128), (513, 17, 64)])
def test_linear_tensor_core_narrow_outputs(M, N, K):
    """N far below the 128-wide tile: the missing weight rows are TMA zero fill, the epilogue writes N columns only."""
    g = torch.Generator().manual_seed(M + N)
    x, w, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / K ** 0.5, torch.randn(N, generator=g)
    y = torch.nn.functional.linear(x.double(), w.double(), b.double())
    out = torch.full((M, N + 3), 7.0, device=DEV)
    ops.linear(x.to(DEV), w.to(DEV), b.to(DEV), out=out[:, :N], precision=1)
    assert float((out[:, :N].cpu().double() - y).abs().max()) < 4e-3 * max(float(y.std()), 1.0)
    assert float((out[:, N:] - 7.0).abs().max()) == 0.0  # nothing written past column N


def test_linear_fp16_split_output():
    """tb_linear Yh: columns >= col_h as fp16 into a second buffer (how the K|V tables of the tensor-core mode are made)."""
    g = torch.Generator().manual_seed(5)
    M, N, K, col_h = 1000, 896, 128, 640
    x, w, b = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / K ** 0.5, torch.randn(N, generator=g)
    y = torch.nn.functional.linear(x.double(), w.double(), b.double())
    yh = torch.full((M, N - col_h + 8), 3.0, dtype=torch.float16, device=DEV)
    y32 = ops.linear(x.to(DEV), w.to(DEV), b.to(DEV), precision=1, out_h=yh[:, :N - col_h], col_h=col_h)
    assert y32.shape == (M, col_h)
    assert float((y32.cpu().double() - y[:, :col_h]).abs().max()) < 4e-3 * float(y.std())
    assert float((yh[:, :N - col_h].cpu().double() - y[:, col_h:]).abs().max()) < 6e-3 * float(y.std())
    assert float((yh[:, N - col_h:].float() - 3.0).abs().max()) == 0.0
    tbl = torch.empty(M, N, dtype=torch.float16, device=DEV)          # col_h = 0: everything fp16, no fp32 output
    assert ops.linear(x.to(DEV), w.to(DEV), b.to(DEV), precision=1, out_h=tbl, col_h=0) is None
    assert float((tbl.cpu().double() - y).abs().max()) < 6e-3 * float(y.std())
    with pytest.raises(RuntimeError):                                  # the fp32 parity path has no fp16 output
        ops.linear(x.to(DEV), w.to(DEV), b.to(DEV), precision=0, out_h=tbl, col_h=0)


@pytest.mark.parametrize("M,N,K,flags", [(1000, 128, 640, "bm"), (4097, 128, 512, "bmr"), (300, 256, 64, "b"), (77, 40, 8, "")])
def test_linear_fp16_operands(M, N, K, flags):
    """tb_linear precision 2: fp16 activations x fp16 weights on tcgen05 kind::f16, fp32 accumulate / bias / residual
    (the consumer of the tensor-core mode's fp16 [ov|z] rows and FFN hidden). The inputs are exactly representable in
    fp16 here, so the result must match the fp64 product to fp32-accumulation accuracy."""
    g = torch.Generator().manual_seed(M + K)
    x = torch.randn(M, K, generator=g).half()
    w = (torch.randn(N, K, generator=g) / K ** 0.5).half()
    b = torch.randn(N, generator=g) if "b" in flags else None
    res = torch.randn(M, N, generator=g) if "r" in flags else None
    mask = torch.rand(M, generator=g) < 0.2 if "m" in flags else None
    y = x.double() @ w.double().t() + (b.double() if b is not None else 0)
    if mask is not None:
        y = y.masked_fill(mask[:, None], 0.0)
    if res is not None:
        y = y + res.double()
    dv = lambda t: None if t is None else t.to(DEV)  # noqa: E731
    out = ops.linear(dv(x), dv(w), dv(b), mask_pre=dv(mask), res=dv(res), precision=2)
    assert float((out.cpu().double() - y).abs().max()) < 2e-5 * max(1.0, float(y.abs().max()))
    with pytest.raises(AssertionError):
        ops.linear(dv(x).float(), dv(w), dv(b), precision=2)


@pytest.mark.parametrize("s", [15, 11, 4, 1])
def test_ag_frontend_fused_vs_oracle(s):
    """tb_ag_frontend (fused history encoder of the tensor-core mode: featurise + input MLP + PoseEmb64 + PointNet on
    mma.sync, fp16 operands) vs the fp32 oracle front-end (agent_encoder.py:130-162) on random ring-buffer states,
    full (s >= W) and partial (s < W) windows, invalid steps and fully invalid agents."""
    from trafficbotsv1_5_b200 import lib as L, config
    from trafficbotsv1_5_b200.model import HotPathModel
    cfg = config.default_model_cfg()
    P = params.init_params(cfg, seed=3)
    m = HotPathModel(P, cfg, config.derived_sizes(cfg), DEV, precision=1)
    W, d, B, A = cfg["temp_window_size"], cfg["hidden_dim"], 3, 37
    g = torch.Generator().manual_seed(100 + s)
    n_step = min(s, W)
    hv = torch.rand(B, A, n_step, generator=g) < 0.8
    hv[0, :3] = False
    hp = torch.cat([(torch.rand(B, A, n_step, 2, generator=g) * 2 - 1) * 120, (torch.rand(B, A, n_step, 1, generator=g) * 2 - 1) * 3], -1)
    hm = torch.cat([torch.rand(B, A, n_step, 1, generator=g) * 20, torch.randn(B, A, n_step, 2, generator=g)], -1)
    attr = torch.cat([torch.rand(B, A, 3, generator=g) * 5, torch.nn.functional.one_hot(torch.randint(0, 3, (B, A), generator=g), 3).float()], -1)
    # oracle (time order, oldest first)
    tok_pose = O.last_valid(hp, hv)
    xy = O.to_local_xy(hp[..., :2], tok_pose[:, :, None, :2], tok_pose[..., 2])
    yaw = hp[..., 2] - tok_pose[..., 2:3]
    rows = torch.cat([attr[:, :, None, :].expand(-1, -1, n_step, -1), hm, torch.eye(W)[None, None, -n_step:].expand(B, A, -1, -1)], -1)
    feat = torch.cat([O.mlp(P, "ag_encoder.input_encoder.mlp", rows, (0, 2, 4), False), O.pose_emb_xy_yaw(xy, yaw, d // 2)], -1)
    ref = O.pointnet(P, "ag_encoder.temp_encoder", feat, ~hv)
    # ring-buffer state: time tau = s - n_step + i lives in slot tau % W
    ring_v = torch.zeros(B, A, W, dtype=torch.uint8)
    ring_p, ring_m = torch.zeros(B, A, W, 3), torch.zeros(B, A, W, 3)
    for i in range(n_step):
        slot = (s - n_step + i) % W
        ring_v[:, :, slot], ring_p[:, :, slot], ring_m[:, :, slot] = hv[:, :, i].to(torch.uint8), hp[:, :, i], hm[:, :, i]
    dv = lambda t: t.to(DEV).contiguous()  # noqa: E731
    blob, bias = m._ag_frontend_weights()
    tok = torch.full((B * A, d + 8), 5.0, device=DEV)
    tp, ti = torch.empty(B, A, 3, device=DEV), torch.empty(B, A, dtype=torch.uint8, device=DEV)
    step = torch.tensor([s], dtype=torch.int32, device=DEV)
    rv, rp, rm, at = dv(ring_v), dv(ring_p), dv(ring_m), dv(attr)
    gen = torch.Generator().manual_seed(s)
    ln_g, ln_b = (torch.rand(d, generator=gen) + 0.5).to(DEV), torch.randn(d, generator=gen).to(DEV)
    ln = torch.full((B * A, d + 8), 7.0, dtype=torch.float16, device=DEV)
    L.check(L.load().tb_ag_frontend(L.ptr(rv), L.ptr(rp), L.ptr(rm), L.ptr(at), L.ptr(step), L.ptr(m.freq_ag), B, A, W,
                                    L.ptr(blob), L.ptr(bias), L.ptr(tok), d + 8, L.ptr(tp), L.ptr(ti), L.ptr(ln_g),
                                    L.ptr(ln_b), L.ptr(ln), d + 8, L.stream()),
            "tb_ag_frontend")
    # the fused first LayerNorm: LayerNorm of the token the kernel wrote, fp16 rows, padding untouched
    ln_ref = torch.nn.functional.layer_norm(tok[:, :d].double(), (d,), ln_g.double(), ln_b.double(), 1e-5)
    assert float((ln[:, :d].double() - ln_ref).abs().max()) < 4e-3 * max(1.0, float(ln_ref.abs().max()))
    assert float((ln[:, d:].float() - 7.0).abs().max()) == 0.0
    assert torch.equal(ti.cpu().bool(), ~hv.any(-1)) and float((tp.cpu() - tok_pose).abs().max()) == 0.0
    out = tok[:, :d].cpu().view(B, A, d)
    scale = float(ref.abs().max())
    err = float((out - ref).abs().max())
    print(f"fused agent front-end s={s}: max err {err:.3e} (scale {scale:.2f})")
    assert err < 2e-3 * scale                       # fp16 operands, 6 layers (measured 4-6e-4)
    assert float(out[0, :3].abs().max()) == 0.0     # agents without a valid step
    assert float((tok[:, d:] - 5.0).abs().max()) == 0.0


@pytest.mark.parametrize("B,S,T0,K0,T1,K1,div1", [(2, 50, 50, 17, 0, 0, 1), (4, 33, 70, 30, 12, 7, 2), (1, 20, 25, 24, 0, 0, 1)])
def test_knarpe_attn_backward_vs_autograd(B, S, T0, K0, T1, K1, div1):
    """SURVEY 8(f) rank 2, first piece: gradient of the KNARPE core (tb_knarpe_attn_bwd) vs torch autograd of the same
    re-associated op in float64 (logits q.k + u.e, base-2 masked softmax, sums of v and e), two K|V tables with
    different batch divisors, masked neighbours, an all-masked token, scatter-add into shared table rows."""
    d = 128
    g = torch.Generator().manual_seed(B * 100 + K0)
    M, K = B * S, K0 + K1
    q = torch.randn(M, d, generator=g) * 0.3
    u = torch.randn(M, H * d, generator=g) * 0.1
    kv0 = torch.randn(B * T0, 2 * d, generator=g)
    kv1 = torch.randn((B // div1) * T1, 2 * d, generator=g) if K1 else None
    idx = torch.cat([torch.stack([torch.randperm(T0, generator=g)[:K0] for _ in range(M)]).view(B, S, K0)] +
                    ([torch.stack([torch.randperm(T1, generator=g)[:K1] for _ in range(M)]).view(B, S, K1)] if K1 else []), -1)
    inv = torch.rand(B, S, K, generator=g) < 0.25
    inv[0, 1] = True
    rel = torch.cat([(torch.rand(B, S, K, 2, generator=g) * 2 - 1) * 100, (torch.rand(B, S, K, 1, generator=g) * 2 - 1) * 3], -1)
    d_out = torch.randn(M, 5 * d, generator=g)

    # float64 autograd reference of the core op (tests/_knarpe_ref.py)
    qd, ud, k0d = q.double().requires_grad_(), u.double().requires_grad_(), kv0.double().requires_grad_()
    k1d = kv1.double().requires_grad_() if K1 else None
    rows = KR.gather_rows(k0d, T0, 1, K0, idx, B, k1d, T1, div1)
    ov, z, _ = KR.knarpe_core(qd, ud, rows, inv, rel)
    out = torch.cat([ov, z], -1)
    out.backward(d_out.double())
    # the forward kernel agrees with this reference (sanity of the test itself)
    dv = lambda t: None if t is None else t.to(DEV).contiguous()  # noqa: E731
    freq = ops.pe_freq_xy(d, 1e3, DEV)
    args = (dv(q), dv(u), dv(kv0), T0, 1, K0, dv(idx.to(torch.int32)), dv(inv), dv(rel), freq, B, S, d)
    fwd, _ = ops.knarpe_attn(*args, kv1=dv(kv1), T1=T1, div1=div1, K1=K1)
    assert rel_l2(fwd, out.detach().float()) < 1e-5
    d_qu, d_kv0, d_kv1 = ops.knarpe_attn_bwd(*args, dv(d_out), kv1=dv(kv1), T1=T1, div1=div1, K1=K1)
    ref_qu = torch.cat([qd.grad, ud.grad], -1).float()
    for name, a, b_ in (("d_q|d_u", d_qu, ref_qu), ("d_kv0", d_kv0, k0d.grad.float())) + \
            ((("d_kv1", d_kv1, k1d.grad.float()),) if K1 else ()):
        err = rel_l2(a, b_)
        print(f"knarpe backward {name}: rel_l2 {err:.2e}")
        assert err < 2e-5, name
    assert float(d_qu.view(B, S, -1)[0, 1].abs().max()) == 0.0  # all-masked token


def test_attention_rpe_dropin_autograd_vs_oracle():
    """Drop-in AttentionRPE with gradients enabled (torch GEMMs + CUDA core forward/backward) vs autograd through the
    oracle restatement of attention_rpe.py:58-198 in float64: output and gradients w.r.t. src, tgt and all six
    parameter tensors (SURVEY 8(f) rank 2: the operator-level piece of the training path)."""
    from trafficbotsv1_5_b200 import reference_api as R
    d, B, S, K = 128, 2, 40, 19
    g = torch.Generator().manual_seed(77)
    shapes = {"in_proj_weight": (3 * d, d), "in_proj_bias": (3 * d,), "out_proj_weight": (d, d), "out_proj_bias": (d,),
              "linear_rpe.weight": (2 * d, d), "linear_rpe.bias": (2 * d,)}
    sd = params.rand_like_state_dict(shapes, 5)
    src, tgt = torch.randn(B, S, d, generator=g), torch.randn(B, S, K, d, generator=g)
    mask = torch.rand(B, S, K, generator=g) < 0.3
    mask[1, 2] = True
    rel = torch.cat([(torch.rand(B, S, K, 2, generator=g) * 2 - 1) * 100, (torch.rand(B, S, K, 1, generator=g) * 2 - 1) * 3], -1)
    G = torch.randn(B, S, d, generator=g)
    # oracle, float64 autograd
    P = {f"a.{k}": v.double().requires_grad_() for k, v in sd.items()}
    s64, t64 = src.double().requires_grad_(), tgt.double().requires_grad_()
    ref = O.attention_rpe(P, "a", s64, t64, mask, O.pose_emb_xy_yaw(rel[..., :2].double(), rel[..., 2].double(), d), H)
    (ref * G.double()).sum().backward()
    # drop-in module on the GPU
    mod = R.AttentionRPE(d, H, dropout_p=0.0, d_rpe=d).to(DEV)
    mod.load_state_dict(sd)
    sg, tg = src.to(DEV).requires_grad_(), tgt.to(DEV).requires_grad_()
    out, _ = mod(sg, tg, mask.to(DEV), None, rel.to(DEV))
    (out * G.to(DEV)).sum().backward()
    assert rel_l2(out.detach(), ref.detach().float()) < 1e-5
    assert float(out.detach()[1, 2].abs().max()) == 0.0
    checks = [("src", sg.grad, s64.grad), ("tgt", tg.grad, t64.grad)] + \
             [(k, dict(mod.named_parameters())[k].grad, P[f"a.{k}"].grad) for k in shapes]
    for name, a, b_ in checks:
        err = rel_l2(a, b_.float())
        print(f"AttentionRPE autograd d/d{name}: rel_l2 {err:.2e}")
        assert err < 5e-5, name
    # inference path of the same module still agrees
    with torch.no_grad():
        out2, _ = mod(src.to(DEV), tgt.to(DEV), mask.to(DEV), None, rel.to(DEV))
    assert rel_l2(out2, ref.detach().float()) < 1e-5


def test_knn_select_temporal_slab_path_exact():
    """tb_knn_select with x-sorted static targets + row_state (the per-step agent -> map select): over a sequence of
    moving / teleporting / invalidated sources the selected SETS, masks and relative poses equal the stateless full
    scan (the slab |x - sx| <= sqrt(kth_prev) + |displacement| always contains the K nearest)."""
    B, S, T, K, div, lim = 6, 70, 1024, 64, 3, 80.0
    g = torch.Generator().manual_seed(11)
    tgt = torch.cat([(torch.rand(B // div, T, 2, generator=g) * 2 - 1) * 150, (torch.rand(B // div, T, 1, generator=g) * 2 - 1) * 3], -1)
    tinv = torch.rand(B // div, T, generator=g) < 0.1
    order = torch.argsort(tgt[..., 0], dim=1)
    s_pose = torch.gather(tgt, 1, order[..., None].expand(-1, -1, 3)).contiguous().to(DEV)
    s_inv = torch.gather(tinv, 1, order).contiguous().to(DEV)
    s_idx = order.to(torch.int32).contiguous().to(DEV)
    state = torch.full((B, S, 3), float("inf"), device=DEV)
    src = torch.cat([(torch.rand(B, S, 2, generator=g) * 2 - 1) * 120, (torch.rand(B, S, 1, generator=g) * 2 - 1) * 3], -1)
    for step in range(8):
        sinv = torch.rand(B, S, generator=g) < 0.1
        if step:
            src = src + torch.cat([torch.randn(B, S, 2, generator=g) * (0.5 + step), torch.randn(B, S, 1, generator=g) * 0.1], -1)
        if step == 4:
            src[:, :10, :2] = (torch.rand(B, 10, 2, generator=g) * 2 - 1) * 140      # teleports
        i0, m0, r0 = ops.knn_select(src.to(DEV), sinv.to(DEV), tgt.to(DEV), tinv.to(DEV), K, lim, tgt_div=div)
        i1, m1, r1 = ops.knn_select(src.to(DEV), sinv.to(DEV), s_pose, s_inv, K, lim, tgt_div=div, index_map=s_idx,
                                    row_state=state, sorted_by_x=True)
        ok = ~sinv.to(DEV)  # rows of invalid sources: fillers only
        o0, o1 = i0.argsort(-1), i1.argsort(-1)
        a0, a1 = torch.gather(i0, 2, o0), torch.gather(i1, 2, o1)
        assert torch.equal(a0[ok], a1[ok]), f"step {step}: selected sets differ"
        assert torch.equal(torch.gather(m0, 2, o0)[ok], torch.gather(m1, 2, o1)[ok])
        rr0 = torch.gather(r0, 2, o0[..., None].expand(-1, -1, -1, 3))[ok]
        rr1 = torch.gather(r1, 2, o1[..., None].expand(-1, -1, -1, 3))[ok]
        assert torch.equal(rr0, rr1)
        assert bool(m1[~ok].all())
    assert bool(torch.isfinite(state[..., 2][ok]).all())  # the fast path was armed


@pytest.mark.parametrize("B,S,K,p_mask", [(3, 33, 25, 0.2), (1, 7, 32, 0.0), (2, 40, 9, 0.5), (1, 64, 25, 0.9), (5, 1, 3, 0.3),
                                          (2, 30, 50, 0.3)])
def test_attention_tensor_core_fp16_operands(B, S, K, p_mask):
    """fp16 [q|u] rows + fp16 K|V tables: lists of <= 32 candidates take the two-tokens-per-warp kernel (odd token
    counts, a single token, empty and ragged lists of the two tokens of a warp), longer ones the one-token kernel."""
    d = 128
    g = torch.Generator().manual_seed(K * 7 + S)
    shapes = {"in_proj_weight": (3 * d, d), "in_proj_bias": (3 * d,), "out_proj_weight": (d, d), "out_proj_bias": (d,),
              "linear_rpe.weight": (2 * d, d), "linear_rpe.bias": (2 * d,)}
    sd = params.rand_like_state_dict(shapes, 23)
    src, tgt = torch.randn(B, S, d, generator=g), torch.randn(B, S, K, d, generator=g)
    mask = torch.rand(B, S, K, generator=g) < p_mask
    mask[0, 0] = True
    if S > 2:
        mask[-1, -2, 1:] = True  # one valid neighbour next to a fuller list
    rel = torch.cat([(torch.rand(B, S, K, 2, generator=g) * 2 - 1) * 300, (torch.rand(B, S, K, 1, generator=g) * 2 - 1) * 3.2], -1)
    P = {f"a.{k}": v for k, v in sd.items()}
    ref = O.attention_rpe(P, "a", src, tgt, mask, O.pose_emb_xy_yaw(rel[..., :2], rel[..., 2], d), H)
    out, nv = _run_attention(sd, src, tgt, mask, rel, half_kv=True, half_qu=True, fast_trig=True)
    scale = float(ref.abs().max())
    err = float((out.cpu() - ref).abs().max()) / scale
    print(f"fp16-operand attention B={B} S={S} K={K}: max err / scale {err:.2e}, rel_l2 {rel_l2(out, ref):.2e}")
    close(out, ref, 4e-3, 4e-3 * scale, "fp16-operand tensor-core attention vs oracle")
    assert rel_l2(out, ref) < 1.5e-3
    assert torch.equal(nv.cpu(), mask.all(-1)) and float(out[0, 0].abs().max()) == 0.0


@pytest.mark.parametrize("B,S,K,p_mask", [(3, 33, 25, 0.2), (1, 7, 32, 0.0), (5, 1, 3, 0.3), (2, 30, 50, 0.3), (2, 21, 128, 0.4)])
def test_attention_head_interleaved_layout_is_bit_identical(B, S, K, p_mask):
    """tb_knarpe_attn flags bit 4: permuting the q / k / v projection features into the head-interleaved order and
    gathering rows with 256-bit loads feeds the MMAs the same fragments -> the same bits as the plain layout."""
    d = 128
    g = torch.Generator().manual_seed(K * 11 + S)
    shapes = {"in_proj_weight": (3 * d, d), "in_proj_bias": (3 * d,), "out_proj_weight": (d, d), "out_proj_bias": (d,),
              "linear_rpe.weight": (2 * d, d), "linear_rpe.bias": (2 * d,)}
    sd = params.rand_like_state_dict(shapes, 29)
    src, tgt = torch.randn(B, S, d, generator=g), torch.randn(B, S, K, d, generator=g)
    mask = torch.rand(B, S, K, generator=g) < p_mask
    mask[0, 0] = True
    rel = torch.cat([(torch.rand(B, S, K, 2, generator=g) * 2 - 1) * 300, (torch.rand(B, S, K, 1, generator=g) * 2 - 1) * 3.2], -1)
    a, nva = _run_attention(sd, src, tgt, mask, rel, half_kv=True, half_qu=True, fast_trig=True)
    b, nvb = _run_attention(sd, src, tgt, mask, rel, half_kv=True, half_qu=True, fast_trig=True, interleaved=True)
    assert torch.equal(a, b) and torch.equal(nva, nvb)
    P = {f"a.{k}": v for k, v in sd.items()}
    ref = O.attention_rpe(P, "a", src, tgt, mask, O.pose_emb_xy_yaw(rel[..., :2], rel[..., 2], d), H)
    close(b, ref, 4e-3, 4e-3 * float(ref.abs().max()), "head-interleaved tensor-core attention vs oracle")


def test_attention_head_interleaved_layout_argument_checks():
    d, B, S, K = 128, 1, 4, 8
    q = torch.zeros(B * S, d + H * d, dtype=torch.float16, device=DEV)
    kv = torch.zeros(B * S * K + 1, 2 * d, dtype=torch.float16, device=DEV)
    idx = torch.zeros(B, S, K, dtype=torch.int32, device=DEV)
    inv = torch.zeros(B, S, K, dtype=torch.bool, device=DEV)
    rel = torch.zeros(B, S, K, 3, device=DEV)
    freq = ops.pe_freq_xy(d, 1e3, DEV)
    with pytest.raises(RuntimeError):  # fp32 q rows: the layout needs flags bits 1 and 3
        ops.knarpe_attn(q[:, :d].float(), q[:, d:].float(), kv, S * K, 1, K, idx, inv, rel, freq, B, S, d, H,
                        interleaved=True, fast_trig=True)
    with pytest.raises(RuntimeError):  # table base only 16-byte aligned
        ops.knarpe_attn(q[:, :d], q[:, d:], kv.view(-1)[8:8 + B * S * K * 2 * d].view(-1, 2 * d), S * K, 1, K, idx, inv,
                        rel, freq, B, S, d, H, interleaved=True, fast_trig=True)


@pytest.mark.parametrize("M,K,extras", [(4096, 640, "mr"), (1000, 512, "rp"), (77, 128, ""), (65536, 640, "mr")])
def test_linear_fused_layernorm(M, K, extras):
    """tb_linear_ln: the projection's fp32 result is bit-identical to tb_linear's, and the fp16 LayerNorm rows written
    by the same epilogue match LayerNorm of that result (eps 1e-5, transformer_rpe.py:156-171) to fp16 rounding.
    Covers full and partial row blocks, residual / pre- and post-masks, many tiles per CTA."""
    N = 128
    g = torch.Generator().manual_seed(M + K)
    x = (torch.randn(M, K, generator=g) * 0.7).half().to(DEV)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).half().to(DEV)
    b = torch.randn(N, generator=g).to(DEV)
    res = (torch.randn(M, N, generator=g) * 2 + 0.5).to(DEV) if "r" in extras else None
    mpre = (torch.rand(M, generator=g) < 0.1).to(DEV) if "m" in extras else None
    mpost = (torch.rand(M, generator=g) < 0.1).to(DEV) if "p" in extras else None
    gamma, beta = (torch.rand(N, generator=g) + 0.5).to(DEV), torch.randn(N, generator=g).to(DEV)
    y0 = ops.linear(x, w, b, mask_pre=mpre, res=res, mask_post=mpost, precision=2)
    y1, ln = ops.linear_ln(x, w, b, gamma, beta, mask_pre=mpre, res=res, mask_post=mpost, precision=2)
    assert torch.equal(y0, y1)
    ref = torch.nn.functional.layer_norm(y1.double(), (N,), gamma.double(), beta.double(), 1e-5)
    err = float((ln.double() - ref).abs().max())
    assert err < 4e-3 * max(1.0, float(ref.abs().max())), err  # fp16 output rounding (2^-11 relative)
    ln2 = ops.layernorm(y1, gamma, beta, out_dtype=torch.float16)
    assert float((ln.float() - ln2.float()).abs().max()) < 4e-3 * max(1.0, float(ref.abs().max()))


def test_linear_fused_layernorm_argument_checks():
    x = torch.zeros(256, 128, dtype=torch.float16, device=DEV)
    g = torch.ones(256, device=DEV)
    with pytest.raises(RuntimeError):  # N != 128
        ops.linear_ln(x, torch.zeros(256, 128, dtype=torch.float16, device=DEV), None, g, g)
    w = torch.zeros(128, 128, dtype=torch.float16, device=DEV)
    with pytest.raises(RuntimeError):  # residual rows only 4-byte aligned
        ops.linear_ln(x, w, None, g[:128], g[:128], res=torch.zeros(256, 132, device=DEV)[:, 1:129])


# ------------------------------------------------------------------------------------------------ fused MLP chain
def _h(t):
    return t.half().float()


@pytest.mark.parametrize("M", [1, 1000, 148 * 3 * 128 + 77])
def test_mlp_chain_program_vs_torch(M):
    """tb_chain_*: a head-chain-shaped program (fp32 LOAD, K = 128 / 256 / 384 GEMM units, ReLU, row masks, fp32 residual,
    in-place units, a 6-wide output) and an FFN-shaped one (fp16 LOAD, 4 hidden units, K = 512, residual, LayerNorm) against
    plain torch on fp16-rounded operands. Error budget: fp16 rounding of every intermediate activation (2^-11 relative)."""
    g = torch.Generator().manual_seed(M)
    d = 128
    rnd = lambda *s, sc=1.0: (torch.randn(*s, generator=g) * sc)  # noqa: E731
    x = rnd(M, 2 * d).to(DEV)                       # x in columns 0..127 of a 256-wide buffer
    ext = rnd(M, d).to(DEV)
    m_pre = (torch.rand(M, generator=g) < 0.3).to(DEV)
    m_post = (torch.rand(M, generator=g) < 0.3).to(DEV)
    W1, b1 = rnd(d, d, sc=0.1), rnd(d, sc=0.1)
    W2, b2 = rnd(d, 2 * d, sc=0.07), rnd(d, sc=0.1)
    W3, b3 = rnd(3 * d, d, sc=0.1), rnd(3 * d, sc=0.1)
    W3b = [rnd(d, d, sc=0.1) for _ in range(3)]
    W4, b4 = rnd(6, 3 * d, sc=0.1), rnd(6, sc=0.1)
    hw = lambda w: w.half().contiguous().to(DEV)  # noqa: E731
    out2 = torch.zeros(M, 2 * d, device=DEV)
    out6 = torch.full((M, 6), 7.0, device=DEV)
    p = ops.ChainProgram(DEV, n_buf=4)
    # bindings: 0 x, 1 ext, 2 m_pre, 3 m_post, 4 out2, 5 out6
    p.load(1, d, 1)
    p.gemm(hw(W1), [1], b1, relu=True, out_buf=2, mask_post=3)
    p.load(0, 2 * d, 0)
    p.gemm(hw(W2), [0, 2], b2, relu=True, mask_pre=2, res=0, ldr=2 * d, out_buf=0, out_g=4, ldg=2 * d, g_col=d)
    for t in range(3):
        p.gemm(hw(W3), [0], b3, n0=t * d, relu=True, out_buf=1 + t)
    for t in range(3):
        p.gemm(hw(W3b[t]), [1 + t], None, relu=True, out_buf=1 + t)  # in place
    p.gemm(hw(W4), [1, 2, 3], b4, out_g=5, ldg=6, n_valid=6)
    p.finish()
    p.run([x, ext, ops._u8(m_pre), ops._u8(m_post), out2, out6], M)
    torch.cuda.synchronize()
    xc, ec = x.cpu(), ext.cpu()
    a1 = torch.relu(_h(ec) @ _h(W1).T + b1).masked_fill(m_post.cpu()[:, None], 0.0)
    cat = torch.cat([_h(xc[:, :d]), _h(a1)], 1)
    x2 = torch.relu(cat @ _h(W2).T + b2).masked_fill(m_pre.cpu()[:, None], 0.0) + xc[:, :d]
    h0 = torch.relu(_h(x2) @ _h(W3).T + b3)
    h1 = torch.cat([torch.relu(_h(h0[:, t * d:(t + 1) * d]) @ _h(W3b[t]).T) for t in range(3)], 1)
    o6 = _h(h1) @ _h(W4).T + b4
    assert float(out2[:, :d].abs().max()) == 0.0                      # untouched columns
    close(out2[:, d:], x2, 2e-3, 2e-3 * float(x2.abs().max()), "chain x2")
    close(out6, o6, 3e-3, 3e-3 * float(o6.abs().max()), "chain 6-wide output")
    # ---- FFN-shaped program: LN rows (fp16) -> linear1 + ReLU (512) -> linear2 + residual + mask -> fp32 out + LN rows
    ln_in = rnd(M, d).half().to(DEV)
    src = rnd(M, d).to(DEV)
    Wa, ba, Wb, bb = rnd(4 * d, d, sc=0.1), rnd(4 * d, sc=0.1), rnd(d, 4 * d, sc=0.05), rnd(d, sc=0.1)
    gam, bet = rnd(d).abs() + 0.5, rnd(d, sc=0.1)
    y = torch.zeros(M, d, device=DEV)
    ln_out = torch.zeros(M, d, dtype=torch.float16, device=DEV)
    q = ops.ChainProgram(DEV, n_buf=5)
    q.load(0, d, 0, f16=True)
    for t in range(4):
        q.gemm(hw(Wa), [0], ba, n0=t * d, relu=True, out_buf=1 + t)
    q.gemm(hw(Wb), [1, 2, 3, 4], bb, res=1, ldr=d, mask_post=2, out_g=3, ldg=d, ln_out=4, ld_ln=d, ln_gamma=gam.to(DEV),
           ln_beta=bet.to(DEV))
    q.finish()
    q.run([ln_in, src, ops._u8(m_post), y, ln_out], M)
    torch.cuda.synchronize()
    hid = torch.relu(ln_in.cpu().float() @ _h(Wa).T + ba)
    yr = (_h(hid) @ _h(Wb).T + bb + src.cpu()).masked_fill(m_post.cpu()[:, None], 0.0)
    close(y, yr, 2e-3, 2e-3 * float(yr.abs().max()), "chain FFN output")
    lnr = torch.nn.functional.layer_norm(yr, (d,), gam, bet, 1e-5)
    live = ~m_post.cpu()
    close(ln_out.float()[live.to(DEV)], lnr[live], 5e-3, 5e-3 * float(lnr.abs().max()), "chain FFN LayerNorm rows")
    # argument checks
    bad = ops.ChainProgram(DEV, n_buf=4)
    bad.gemm(hw(W1), [1], b1, out_buf=2)  # reads a buffer nobody wrote
    with pytest.raises(RuntimeError):
        bad.finish()


# ------------------------------------------------------------------------------------------------ plain entry points
def test_colsum_accumulates_column_sums():
    """tb_colsum (bias gradient): out[n] += sum_m X[m, n] on a strided view, accumulated into a pre-filled buffer."""
    from trafficbotsv1_5_b200 import lib as L
    g = torch.Generator().manual_seed(9)
    x = torch.randn(70001, 200, generator=g).to(DEV)
    xv = x[:, 8:8 + 130]
    out = torch.full((130,), 3.0, device=DEV)
    L.check(L.load().tb_colsum(L.ptr(xv), xv.stride(0), xv.shape[0], 130, L.ptr(out), L.stream()), "tb_colsum")
    ref = 3.0 + xv.double().sum(0)
    assert float((out.double() - ref).abs().max()) < 1e-5 * float(xv.abs().sum(0).max())


def test_featurize_shared_counter_entry_points_match_per_row_counters():
    """tb_ag_featurize / tb_tl_featurize (one device-side loop counter for the whole batch) are the step_stride = 0 case
    of the *_ex entry points: a batch whose rows all carry the same counter must produce identical bytes either way."""
    from trafficbotsv1_5_b200 import lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(4)
    B, A, TL, W, s = 6, 9, 5, 11, 14
    hv = (torch.rand(B, A, W, generator=g) < 0.8).to(torch.uint8).to(DEV)
    hp = (torch.randn(B, A, W, 3, generator=g) * 20).to(DEV)
    hm = torch.randn(B, A, W, 3, generator=g).to(DEV)
    attr = torch.rand(B, A, 6, generator=g).to(DEV)
    freq = ops.pe_freq_xy(64, 1e3, DEV)
    d1 = torch.tensor([s], dtype=torch.int32, device=DEV)
    dB = torch.full((B,), s, dtype=torch.int32, device=DEV)

    def ag(ex):
        o = dict(pose=torch.zeros(B, A, 3, device=DEV), inv=torch.zeros(B, A, dtype=torch.uint8, device=DEV),
                 rinv=torch.zeros(B, A, W, dtype=torch.uint8, device=DEV), attr=torch.zeros(B * A * W, 9 + W, device=DEV),
                 pe=torch.zeros(B * A * W, 64, device=DEV))
        tail = (L.ptr(freq), B, A, W, L.ptr(o["pose"]), L.ptr(o["inv"]), L.ptr(o["rinv"]), L.ptr(o["attr"]), 9 + W,
                L.ptr(o["pe"]), 64, L.stream())
        if ex:
            L.check(lib.tb_ag_featurize_ex(L.ptr(hv), L.ptr(hp), L.ptr(hm), L.ptr(attr), L.ptr(dB), 1, *tail), "ag_ex")
        else:
            L.check(lib.tb_ag_featurize(L.ptr(hv), L.ptr(hp), L.ptr(hm), L.ptr(attr), L.ptr(d1), *tail), "ag")
        return o

    a, b = ag(False), ag(True)
    for k in a:
        assert torch.equal(a[k], b[k]), k
    assert float(a["pe"].abs().sum()) > 0 and int(a["rinv"].sum()) > 0

    ht = torch.nn.functional.one_hot(torch.randint(0, 5, (B, TL, W), generator=g), 5).to(torch.uint8).to(DEV)
    tinv = (torch.rand(B, TL, generator=g) < 0.2).to(torch.uint8).to(DEV)

    def tl(ex):
        rows, rinv = torch.zeros(B * TL * W, 16, device=DEV), torch.zeros(B, TL, W, dtype=torch.uint8, device=DEV)
        if ex:
            L.check(lib.tb_tl_featurize_ex(L.ptr(ht), L.ptr(tinv), L.ptr(dB), 1, B, TL, W, L.ptr(rows), 16, L.ptr(rinv),
                                           L.stream()), "tl_ex")
        else:
            L.check(lib.tb_tl_featurize(L.ptr(ht), L.ptr(tinv), L.ptr(d1), B, TL, W, L.ptr(rows), 16, L.ptr(rinv),
                                        L.stream()), "tl")
        return rows, rinv

    (r0, i0), (r1, i1) = tl(False), tl(True)
    assert torch.equal(r0, r1) and torch.equal(i0, i1) and float(r0.sum()) > 0
