"""Float64 reference of the KNARPE attention core (tb_knarpe_attn / tb_knarpe_attn_bwd), shared by the GPU tests.

The core is the re-associated attention of DESIGN.md §3 between the projections: per token m and head h

    logit[m, h, j] = q[m, h] . k[row(m, j), h] + u[m, h] . e[m, j]      (log2 units, scale folded into q and u)
    p = base-2 softmax over the unmasked neighbours j
    ov[m, h] = sum_j p v[row(m, j), h]        z[m, h] = sum_j p e[m, j]

with e = PoseEmb(rel) (utils/pose_emb.py:50-55). A token whose neighbours are all masked gets ov = z = 0 and
none_valid = True (attention_rpe.py:188-190). Everything runs in the dtype of the inputs (float64 for the tests), so
it is differentiable with torch autograd."""
import math

import torch

from oracle import tb_oracle as O


def gather_rows(kv0, T0, div0, K0, idx, B, kv1=None, T1=0, div1=1):
    """K|V rows of every (token, neighbour): idx[..., :K0] index table 0 of scene b // div0, idx[..., K0:] table 1 of
    scene b // div1. kv tables are [n_tables * T, 2d] (any row stride); returns [B, S, K, 2d]."""
    bs = torch.arange(B)
    rows = kv0.reshape(-1, T0, kv0.shape[-1])[(bs // div0)[:, None, None], idx[..., :K0].long()]
    if idx.shape[-1] > K0:
        rows1 = kv1.reshape(-1, T1, kv1.shape[-1])[(bs // div1)[:, None, None], idx[..., K0:].long()]
        rows = torch.cat([rows, rows1], 2)
    return rows


def knarpe_core(q, u, rows, inv, rel=None, emb=None, n_head=4):
    """q [M, d], u [M, H*d], rows [B, S, K, 2d] (gather_rows), inv [B, S, K] (True = masked), exactly one of rel
    [B, S, K, 3] (embedding evaluated here, in the dtype of q) or emb [B, S, K, d].
    Returns ov [M, d], z [M, H*d], none_valid [M]."""
    B, S, K, d2 = rows.shape
    d, H, M = d2 // 2, n_head, B * S
    dh = d // H
    if emb is None:
        emb = O.pose_emb_xy_yaw(rel[..., :2].to(q.dtype), rel[..., 2].to(q.dtype), d)
    e = emb.to(q.dtype).reshape(M, K, d)
    kk, vv = rows[..., :d].reshape(M, K, H, dh), rows[..., d:].reshape(M, K, H, dh)
    lg = torch.einsum("mhc,mkhc->mhk", q.reshape(M, H, dh), kk) + torch.einsum("mhc,mkc->mhk", u.reshape(M, H, d), e)
    msk = inv.reshape(M, 1, K)
    none = inv.reshape(M, K).all(-1)
    p = torch.softmax((lg * math.log(2.0)).masked_fill(msk, -float("inf")).masked_fill(none[:, None, None], 0.0), -1)
    p = p.masked_fill(msk, 0.0)
    ov = torch.einsum("mhk,mkhc->mhc", p, vv).reshape(M, d)
    z = torch.einsum("mhk,mkc->mhc", p, e).reshape(M, H * d)
    return ov.masked_fill(none[:, None], 0.0), z.masked_fill(none[:, None], 0.0), none


def attention_from_core(fused, src, tgt, mask, rel, n_head=4):
    """AttentionRPE (attention_rpe.py:58-198, RPE branch) composed from the core and the packed projections of
    model.fuse_attention: [q|u] = in-projection of src, K|V table = projection of the gathered tgt rows
    (table = tgt flattened, idx = s*K + k), output = out-projection of [ov|z], all-masked tokens zero."""
    B, S, K, d = tgt.shape
    f = {k: v.to(src.dtype) for k, v in fused.items()}
    qu = src.reshape(B * S, d) @ f["w_in_q"].T + f["b_in_q"]
    kv = tgt.reshape(B * S * K, d) @ f["w_kv"].T + f["b_kv"]
    idx = torch.arange(S * K).view(1, S, K).expand(B, -1, -1)
    ov, z, none = knarpe_core(qu[:, :d], qu[:, d:], gather_rows(kv, S * K, 1, K, idx, B), mask, rel, n_head=n_head)
    out = torch.cat([ov, z], -1) @ f["w_out"].T + f["b_out"]
    return out.masked_fill(none[:, None], 0.0).view(B, S, d)
