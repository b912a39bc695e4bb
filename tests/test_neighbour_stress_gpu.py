"""Stress tests of the two neighbour kernels of every policy step against plain float64 references: the KNARPE attention
core (tb_knarpe_attn, tb_knarpe_attn_bwd) at controlled, peaked logits, and the KNN select (tb_knn_select) on exact
integer geometry with exact distance ties.

Attention core
--------------
Every case uses one K|V row per (token, neighbour) (T0 = S*K, idx = s*K + k), so the logit of each (token, head,
neighbour) can be set directly: q_h is random with |q_h| ~ 1, k_hj = l_hj q_h / |q_h|^2 plus noise orthogonal to q_h,
and u is small (u.e ~ 0.2) so that the 16-bit rounding of the embedding does not grow with the logit spread. The
schedules l_hj (log2 units) are mixed across the heads of a token, so a head-slot mix-up shows:
  asc0.5 / asc1.2 / asc3   l_j = a (j - K + 1): the maximum moves up in every group of neighbours. The pair kernel
                           re-establishes its lazy maximum only when a logit beats it by more than 8: with a = 1.2 every
                           8-row group does (9.6), with 0.5 every few groups; a = 3 underflows the early p to 0.
  desc                     l_j = -1.2 j: the maximum is in the first group, no rescale ever runs.
  spike_last / spike_mid   +40 on one neighbour (last, middle) of a 0.5-sigma background; masked neighbours in front
                           of the middle one move it between groups when the list is compacted.
  low                      everything around -60.
Tokens 0-3 (the first two token pairs of the pair kernel) carry opposite schedules and unequal lists: token 0 all
valid ascending vs token 1 with 3 valid descending, token 2 with none valid vs token 3 all valid.

The reference (tests/_knarpe_ref.py) reads exactly what the kernel reads: for 16-bit paths the fp16-rounded q, u, k,
v. Tolerances, each on ov and z separately and relative to each one's own scale (max |ref|):
  fp32 paths   rel-L2 <= 1e-5 (the backward test's bound). The dominant error is the fp32 logit: the q.k sum of
               terms of one sign rounds to <= |l| 2^-24 (log2(d_head) + 1) ~ 2e-6 relative to l at |l| <= 60 near the
               maximum; the fast-trig paths run on |angle| <= 32 rad, where the SFU error is <= 32 2^-22 = 7.6e-6.
  16-bit paths 4e-3 of scale per element and 1.5e-3 rel-L2 (the stated 16-bit tolerances): p and e are rounded to
               fp16 (2^-11 relative), the outputs of fp16 rows too.
none_valid must be exact, and tokens without a valid neighbour exactly 0.

Dispatch matrix of tb_knarpe_attn (csrc/knarpe_attn.cu:356-415); every row is one kernel instantiation and runs in
test_dispatch_matrix with the asc1.2 schedule:
  kv    q     out   D    list    rel/emb  fast_trig  il | kernel
  f16   f16   f16   128  <= 128  rel      ignored    0  | knarpe_attn_mma_pair_kernel<OUT_H=1, IL=0>
  f16   f16   f16   128  <= 128  rel      ignored    1  | knarpe_attn_mma_pair_kernel<1, 1>
  f16   f16   f32   128  <= 128  rel      ignored    0  | knarpe_attn_mma_pair_kernel<0, 0>
  f16   f16   f32   128  <= 128  rel      ignored    1  | knarpe_attn_mma_pair_kernel<0, 1>
  f16   f16   f16   128  > 128   rel      1          0  | knarpe_attn_kernel<128, rel, fast, OUT_H, IN_H, KV_H>
  f16   f32   f32   128  any     rel      1          0  | knarpe_attn_kernel<128, rel, fast, KV_H>
  f16   f16   f16   256  any     rel      1          0  | knarpe_attn_kernel<256, rel, fast, OUT_H, IN_H, KV_H>
  f16   f32   f32   256  any     rel      1          0  | knarpe_attn_kernel<256, rel, fast, KV_H>
  f32   f16   f16   128  any     rel      1          0  | knarpe_attn_kernel<128, rel, fast, OUT_H, IN_H>
  f32   f32   f16   128  any     rel      1          0  | knarpe_attn_kernel<128, rel, fast, OUT_H>
  f32   f32   f32   128  any     emb      ignored    0  | knarpe_attn_kernel<128, emb, exact>
  f32   f32   f32   128  any     rel      1          0  | knarpe_attn_kernel<128, rel, fast>
  f32   f32   f32   128  any     rel      0          0  | knarpe_attn_kernel<128, rel, exact>
  f32   f32   f32   256  any     emb      ignored    0  | knarpe_attn_kernel<256, emb, exact>
  f32   f32   f32   256  any     rel      1          0  | knarpe_attn_kernel<256, rel, fast>
  f32   f32   f32   256  any     rel      0          0  | knarpe_attn_kernel<256, rel, exact>
Every other combination is refused with "unsupported size" (test_dispatch_refusals).

KNN select
----------
Targets sit on an integer grid in [-40, 40]^2 (each pose repeated 1-4 times, some invalid), sources at integer points
with yaw 0. Squared distances are then exact in fp32 and float64 and the rotation into the source frame is exact, so
the tie classes are the true ones and the selection is fully determined: the first K of a stable sort by (distance,
index), emitted in ascending index order, with exact invalid flags (d > dist_limit, targets at exactly the limit
included) and exact relative poses.
"""
import math

import pytest
import torch

import _knarpe_ref as KR

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from trafficbotsv1_5_b200 import ops
    from trafficbotsv1_5_b200.model import head_interleave_perm

DEV = "cuda"
H = 4
SCHED = ["asc1.2", "desc", "spike_last", "asc0.5", "low", "spike_mid", "asc3"]


# ------------------------------------------------------------------------------------------------ attention: inputs
def _sched(kind, K, g):
    j = torch.arange(K, dtype=torch.float64)
    if kind.startswith("asc"):
        return float(kind[3:]) * (j - (K - 1))
    if kind == "desc":
        return -1.2 * j
    noise = 0.5 * torch.randn(K, generator=g, dtype=torch.float64)
    if kind == "spike_last":
        noise[K - 1] += 40.0
        return noise
    if kind == "spike_mid":
        noise[K // 2] += 40.0
        return noise
    assert kind == "low"
    return noise - 60.0


def _logits(M, K, g, scheds):
    """[M, H, K] logits: head h of token m follows scheds[(m + h) % len]; tokens 0-3 as in the module docstring."""
    ell = torch.stack([torch.stack([_sched(scheds[(m + h) % len(scheds)], K, g) for h in range(H)]) for m in range(M)])
    if M >= 4 and len(scheds) > 1:
        ell[0] = _sched("asc1.2", K, g)
        ell[1] = _sched("asc1.2", K, g).flip(0)
        ell[2] = _sched("desc", K, g)
        ell[3] = _sched("asc1.2", K, g)
    return ell


def _mask(B, S, K, g, p_mask, special):
    mask = torch.rand(B, S, K, generator=g) < p_mask
    mask[..., K // 2] = False  # spike neighbours stay valid (the ones in front of the middle spike may be masked)
    mask[..., K - 1] = False
    if special and B * S >= 4:
        m = mask.view(B * S, K)
        m[0] = False
        m[1] = True
        m[1, torch.tensor([0, K // 2, K - 1])] = False  # 3 valid (fewer if K < 3)
        m[2] = True
        m[3] = False
    return mask


def _controlled(B, S, K, D, seed, p_mask=0.2, scheds=SCHED, xy=50.0, yaw=3.0, K0=None):
    """Inputs with the logits of _logits. Returns a dict of fp32 CPU tensors: q [M, D], u [M, H*D], rows [B, S, K, 2D]
    (the K|V row of every (token, neighbour)), inv, rel, and the split K0 of the list into two tables."""
    g = torch.Generator().manual_seed(seed)
    M, dh = B * S, D // H
    ell = _logits(M, K, g, scheds)
    q = torch.randn(M, H, dh, generator=g, dtype=torch.float64) / math.sqrt(dh)
    qq = (q * q).sum(-1, keepdim=True)
    noise = 0.3 * torch.randn(M, H, K, dh, generator=g, dtype=torch.float64) / math.sqrt(dh)
    noise = noise - (noise * q[:, :, None]).sum(-1, keepdim=True) / qq[:, :, None] * q[:, :, None]
    k = ell[..., None] * (q / qq)[:, :, None] + noise                                   # [M, H, K, dh]
    v = torch.randn(M, K, D, generator=g, dtype=torch.float64)
    u = 0.02 * torch.randn(M, H * D, generator=g, dtype=torch.float64)
    rows = torch.cat([k.permute(0, 2, 1, 3).reshape(M, K, D), v], -1).view(B, S, K, 2 * D)
    rel = torch.cat([(torch.rand(B, S, K, 2, generator=g) * 2 - 1) * xy, (torch.rand(B, S, K, 1, generator=g) * 2 - 1) * yaw], -1)
    return dict(q=q.reshape(M, D).float(), u=u.float(), rows=rows.float(), inv=_mask(B, S, K, g, p_mask, len(scheds) > 1),
                rel=rel, B=B, S=S, K=K, D=D, K0=K if K0 is None else K0)


def _run(c, kv_dtype, q_dtype, out_dtype, fast_trig=True, il=False, use_emb=False):
    """Runs tb_knarpe_attn on case c; returns (out [M, D + H*D] on the CPU as float64, none_valid, ref ov, ref z, ref
    none_valid), the reference reading the kernel's (rounded) inputs."""
    B, S, K, D, K0 = c["B"], c["S"], c["K"], c["D"], c["K0"]
    K1 = K - K0
    q, u, rows = c["q"].to(q_dtype), c["u"].to(q_dtype), c["rows"].to(kv_dtype)
    # two tables when K1 > 0: neighbours < K0 read table 0 ([B*S*K0] rows), the others table 1 ([B*S*K1] rows)
    tab0 = rows[:, :, :K0].reshape(-1, 2 * D).contiguous()
    tab1 = rows[:, :, K0:].reshape(-1, 2 * D).contiguous() if K1 else None
    idx = torch.cat([torch.arange(S * K0).view(S, K0)] + ([torch.arange(S * K1).view(S, K1)] if K1 else []), -1)
    idx = idx.to(torch.int32).view(1, S, K).expand(B, -1, -1).contiguous()
    emb = None
    if use_emb:
        from oracle import tb_oracle as O
        emb = O.pose_emb_xy_yaw(c["rel"][..., :2], c["rel"][..., 2], D).contiguous()
    ref_ov, ref_z, ref_none = KR.knarpe_core(q.double(), u.double(), KR.gather_rows(
        tab0.double(), S * K0, 1, K0, idx, B, tab1.double() if K1 else None, S * K1, 1), c["inv"],
        rel=None if use_emb else c["rel"].double(), emb=emb.double() if use_emb else None)
    qd, t0d, t1d = q, tab0, tab1
    if il:  # head-interleaved q / K / V channels (tb_knarpe_attn flags bit 4); ov / z stay in the plain order
        perm = head_interleave_perm(D)
        qd = q[:, perm]
        t0d = torch.cat([tab0[:, :D][:, perm], tab0[:, D:][:, perm]], 1)
        t1d = torch.cat([tab1[:, :D][:, perm], tab1[:, D:][:, perm]], 1) if K1 else None
    dv = lambda t: None if t is None else t.contiguous().to(DEV)  # noqa: E731
    out, nv = ops.knarpe_attn(dv(qd), dv(u), dv(t0d), S * K0, 1, K0, dv(idx), dv(c["inv"]),
                              None if use_emb else dv(c["rel"]), ops.pe_freq_xy(D, 1e3, DEV), B, S, D, H,
                              kv1=dv(t1d), T1=S * K1, div1=1, K1=K1, emb=dv(emb), fast_trig=fast_trig, interleaved=il,
                              out_dtype=out_dtype)
    return out.cpu().double(), nv.cpu(), ref_ov, ref_z, ref_none


def _rel_l2(a, b):
    return float((a - b).norm() / b.norm().clamp(min=1e-300))


def _check(res, sixteen, what):
    out, nv, ref_ov, ref_z, ref_none = res
    D = ref_ov.shape[1]
    assert torch.equal(nv, ref_none), f"{what}: none_valid"
    assert bool((out[ref_none] == 0).all()), f"{what}: tokens without a valid neighbour must be exactly 0"
    for name, a, b in (("ov", out[:, :D], ref_ov), ("z", out[:, D:], ref_z)):
        scale = float(b.abs().max())
        err, l2 = float((a - b).abs().max()) / scale, _rel_l2(a, b)
        print(f"{what} {name}: max err / scale {err:.2e}, rel-L2 {l2:.2e}")
        if sixteen:
            assert err <= 4e-3 and l2 <= 1.5e-3, f"{what} {name}: max err / scale {err:.2e}, rel-L2 {l2:.2e}"
        else:
            assert l2 <= 1e-5, f"{what} {name}: rel-L2 {l2:.2e}"


# ------------------------------------------------------------------------------------------------ attention: tests
@pytest.mark.parametrize("K", [1, 8, 9, 25, 64, 89, 127, 128])
def test_pair_kernel_peaked_logits(K):
    """fp16 q / u / tables, fp16 [ov|z]: the pair kernel (two tokens per warp) at every schedule; K = 89 is two lists
    (64 + 25, the agent -> map / traffic-light shape). B = 3 x S = 21 tokens: a token pair straddles a scene boundary
    and the last token has no partner."""
    c = _controlled(3, 21, K, 128, seed=1000 + K, K0=64 if K == 89 else None)
    _check(_run(c, torch.float16, torch.float16, torch.float16), True, f"pair K={K}")


@pytest.mark.parametrize("K", [129, 160])
def test_simt_fp16_tables_long_lists_peaked_logits(K):
    """Lists over 128 on fp16 tables with fp16 q / u / outputs: the SIMT kernel with KV_H, IN_H and OUT_H."""
    c = _controlled(2, 13, K, 128, seed=2000 + K)
    _check(_run(c, torch.float16, torch.float16, torch.float16), True, f"simt fp16 K={K}")


@pytest.mark.parametrize("D", [128, 256])
def test_simt_fp32_peaked_logits(D):
    """fp32 tables, q / u and outputs, exact trig: the SIMT kernel's per-group rescale with corrections far from 1,
    different for each head slot (slot i of a lane holds head i ^ (lane >> 3))."""
    c = _controlled(2, 11, 70, D, seed=3000 + D)
    _check(_run(c, torch.float32, torch.float32, torch.float32, fast_trig=False), False, f"simt fp32 D={D}")


# kv, q, out dtypes ('h' fp16, 'f' fp32), D, K, use_emb, fast_trig, il: one row per kernel instantiation (docstring)
DISPATCH = [
    ("h", "h", "h", 128, 40, False, True, False), ("h", "h", "h", 128, 40, False, True, True),
    ("h", "h", "f", 128, 40, False, False, False), ("h", "h", "f", 128, 40, False, True, True),
    ("h", "h", "h", 128, 150, False, True, False), ("h", "f", "f", 128, 40, False, True, False),
    ("h", "h", "h", 256, 40, False, True, False), ("h", "f", "f", 256, 40, False, True, False),
    ("f", "h", "h", 128, 40, False, True, False), ("f", "f", "h", 128, 40, False, True, False),
    ("f", "f", "f", 128, 40, True, False, False), ("f", "f", "f", 128, 40, False, True, False),
    ("f", "f", "f", 128, 40, False, False, False), ("f", "f", "f", 256, 40, True, False, False),
    ("f", "f", "f", 256, 40, False, True, False), ("f", "f", "f", 256, 40, False, False, False),
]
_DT = {"h": torch.float16, "f": torch.float32}


@pytest.mark.parametrize("kv,qd,od,D,K,use_emb,fast,il", DISPATCH)
def test_dispatch_matrix(kv, qd, od, D, K, use_emb, fast, il):
    sixteen = "h" in (kv, qd, od)
    # fp32 fast-trig paths: angles within +-32 rad (module docstring)
    xy, yaw = (50.0, 3.0) if (sixteen or not fast) else (2.0, 0.5)
    c = _controlled(3, 9, K, D, seed=4000 + D + K, scheds=["asc1.2"], xy=xy, yaw=yaw)
    c["inv"].view(-1, K)[4] = True  # one token without a valid neighbour
    _check(_run(c, _DT[kv], _DT[qd], _DT[od], fast_trig=fast, il=il, use_emb=use_emb), sixteen,
           f"dispatch kv={kv} q={qd} out={od} D={D} K={K} emb={use_emb} fast={fast} il={il}")


# kv, q, out, D, K, use_emb, fast_trig, il, why
REFUSED = [
    ("h", "h", "h", 128, 40, True, True, False, "fp16 tables need rel (no materialised embedding)"),
    ("h", "f", "f", 128, 40, False, True, True, "interleaved layout with fp32 q / u"),
    ("h", "h", "h", 128, 150, False, True, True, "interleaved layout on the SIMT kernel (list > 128)"),
    ("h", "h", "h", 256, 40, False, False, False, "SIMT kernel on fp16 tables without fast trig"),
    ("h", "f", "h", 128, 40, False, True, False, "fp32 q / u with fp16 outputs on fp16 tables"),
    ("h", "h", "f", 256, 40, False, True, False, "fp16 q / u with fp32 outputs on the SIMT fp16-table kernel"),
    ("f", "f", "f", 128, 40, False, True, True, "interleaved layout on fp32 tables"),
    ("f", "h", "f", 128, 40, False, True, False, "fp16 q / u with fp32 outputs on fp32 tables"),
    ("f", "f", "h", 256, 40, False, True, False, "16-bit rows at D = 256 on fp32 tables"),
    ("f", "f", "h", 128, 40, True, True, False, "16-bit rows with a materialised embedding"),
    ("f", "f", "h", 128, 40, False, False, False, "16-bit rows without fast trig"),
]


@pytest.mark.parametrize("kv,qd,od,D,K,use_emb,fast,il,why", REFUSED)
def test_dispatch_refusals(kv, qd, od, D, K, use_emb, fast, il, why):
    c = _controlled(1, 4, K, D, seed=5, scheds=["asc1.2"])
    with pytest.raises(RuntimeError, match="unsupported"):
        _run(c, _DT[kv], _DT[qd], _DT[od], fast_trig=fast, il=il, use_emb=use_emb)


def test_dispatch_refuses_other_head_counts_and_widths():
    for D, Hh in ((128, 8), (64, 4)):
        q = torch.zeros(8, D * (Hh + 1), device=DEV)
        kv = torch.zeros(8 * 4, 2 * D, device=DEV)
        idx = torch.zeros(1, 8, 4, dtype=torch.int32, device=DEV)
        inv = torch.zeros(1, 8, 4, dtype=torch.bool, device=DEV)
        rel = torch.zeros(1, 8, 4, 3, device=DEV)
        with pytest.raises(RuntimeError, match="unsupported"):
            ops.knarpe_attn(q[:, :D], q[:, D:], kv, 32, 1, 4, idx, inv, rel, ops.pe_freq_xy(128, 1e3, DEV), 1, 8, D, Hh)


@pytest.mark.parametrize("R,div1", [(4, 2), (3, 1)])
@pytest.mark.parametrize("il", [False, True])
@pytest.mark.parametrize("out_dtype", [torch.float16, torch.float32])
def test_pair_kernel_engine_layout(R, div1, il, out_dtype):
    """The engine's configuration of the pair kernel (model.py:227-257, 619-621): B = 2 scenes x R rollouts, S = 37
    agents (odd, so token pairs straddle scene boundaries), one fp16 row buffer [q | u | k | v] of 896 halves per token.
    Self-attention reads q / u / k|v as strided views of that buffer (k|v at column 640, table = the scene's own rows);
    the cross-attention reads q / u from the same buffer and two tables: map rows K0 = 64 with div0 = R, traffic-light
    rows K1 = 25 with div1. With R = 3 / div1 = 1 the pairs also straddle the boundaries of both cross tables."""
    d, B, S, n_mp, n_tl = 128, 2 * R, 37, 300, 40
    M = B * S
    g = torch.Generator().manual_seed(7 * R + div1 + 2 * il)
    buf = torch.zeros(M, 896, dtype=torch.float16)
    buf[:, :d] = (torch.randn(M, d, generator=g) * 0.6).half()
    buf[:, d:5 * d] = (torch.randn(M, 4 * d, generator=g) * 0.02).half()
    buf[:, 5 * d:] = torch.randn(M, 2 * d, generator=g).half()
    mp = torch.randn((B // R) * n_mp, 2 * d, generator=g).half()
    tl = torch.randn((B // div1) * n_tl, 2 * d, generator=g).half()

    def lists(K, T):
        idx = torch.stack([torch.randperm(T, generator=g)[:K] for _ in range(M)]).view(B, S, K).to(torch.int32)
        inv = torch.rand(B, S, K, generator=g) < 0.2
        rel = torch.cat([(torch.rand(B, S, K, 2, generator=g) * 2 - 1) * 80, (torch.rand(B, S, K, 1, generator=g) * 2 - 1) * 3], -1)
        return idx, inv, rel

    si, sinv, srel = lists(25, S)
    sinv.view(M, 25)[S] = True  # the first token of scene-rollout 1 (token B of a straddling pair): nothing valid
    ci, cinv, crel = lists(89, n_mp)
    ci[..., 64:] = torch.randint(0, n_tl, (B, S, 25), generator=g, dtype=torch.int32)
    cinv.view(M, 89)[2 * S - 1] = True

    perm = head_interleave_perm(d) if il else torch.arange(d)
    dbuf = buf.clone()
    for c0 in (0, 5 * d, 6 * d):  # q, k, v channels in the layout the kernel reads
        dbuf[:, c0:c0 + d] = buf[:, c0:c0 + d][:, perm]
    dmp = torch.cat([mp[:, :d][:, perm], mp[:, d:][:, perm]], 1)
    dtl = torch.cat([tl[:, :d][:, perm], tl[:, d:][:, perm]], 1)
    dv = lambda t: t.contiguous().to(DEV)  # noqa: E731
    gb, gmp, gtl = dv(dbuf), dv(dmp), dv(dtl)
    freq = ops.pe_freq_xy(d, 1e3, DEV)
    kw = dict(fast_trig=True, interleaved=il, out_dtype=out_dtype)
    o_self, nv_self = ops.knarpe_attn(gb[:, :d], gb[:, d:5 * d], gb[:, 5 * d:], S, 1, 25, dv(si), dv(sinv), dv(srel),
                                      freq, B, S, d, H, **kw)
    o_x, nv_x = ops.knarpe_attn(gb[:, :d], gb[:, d:5 * d], gmp, n_mp, R, 64, dv(ci), dv(cinv), dv(crel), freq, B, S, d,
                                H, kv1=gtl, T1=n_tl, div1=div1, K1=25, **kw)
    q, u = buf[:, :d].double(), buf[:, d:5 * d].double()
    ref_self = KR.knarpe_core(q, u, KR.gather_rows(buf[:, 5 * d:].double(), S, 1, 25, si, B), sinv, srel.double())
    ref_x = KR.knarpe_core(q, u, KR.gather_rows(mp.double(), n_mp, R, 64, ci, B, tl.double(), n_tl, div1), cinv,
                           crel.double())
    _check((o_self.cpu().double(), nv_self.cpu()) + ref_self, True, f"engine self R={R} il={il} {out_dtype}")
    _check((o_x.cpu().double(), nv_x.cpu()) + ref_x, True, f"engine cross R={R} div1={div1} il={il} {out_dtype}")


@pytest.mark.parametrize("sched", ["asc1.2", "asc3", "spike_last", "spike_mid"])
def test_backward_peaked_logits(sched):
    """tb_knarpe_attn_bwd (exact maximum, knarpe_attn_bwd.cu:124-140) vs float64 autograd of the same reference at the
    existing 2e-5 rel-L2, on peaked schedules (one schedule for all heads, plus the mixed tokens 0-3)."""
    B, S, K, D = 2, 17, 40, 128
    c = _controlled(B, S, K, D, seed=6000 + len(sched), scheds=[sched, "desc"], xy=50.0, yaw=3.0)
    M = B * S
    g = torch.Generator().manual_seed(61)
    d_out = torch.randn(M, 5 * D, generator=g)
    tab = c["rows"].reshape(-1, 2 * D).contiguous()
    idx = torch.arange(S * K, dtype=torch.int32).view(1, S, K).expand(B, -1, -1).contiguous()
    qd, ud, kd = (t.double().requires_grad_() for t in (c["q"], c["u"], tab))
    ov, z, _ = KR.knarpe_core(qd, ud, KR.gather_rows(kd, S * K, 1, K, idx, B), c["inv"], c["rel"])
    torch.cat([ov, z], -1).backward(d_out.double())
    dv = lambda t: t.contiguous().to(DEV)  # noqa: E731
    args = (dv(c["q"]), dv(c["u"]), dv(tab), S * K, 1, K, dv(idx), dv(c["inv"]), dv(c["rel"]), ops.pe_freq_xy(D, 1e3, DEV),
            B, S, D)
    d_qu, d_kv, _ = ops.knarpe_attn_bwd(*args, dv(d_out))
    for name, a, b in (("d_q", d_qu[:, :D], qd.grad), ("d_u", d_qu[:, D:], ud.grad), ("d_kv", d_kv, kd.grad)):
        err = _rel_l2(a.cpu().double(), b)
        print(f"backward {sched} {name}: rel-L2 {err:.2e}")
        assert err < 2e-5, (sched, name, err)


# ------------------------------------------------------------------------------------------------ KNN select
def _grid_targets(Bt, T, g, p_inv=0.15, lo=-40, hi=40):
    """[Bt, T, 3] integer-grid targets, each (x, y) repeated 1-4 times at shuffled positions; random yaw."""
    pose = torch.empty(Bt, T, 3)
    for b in range(Bt):
        pts = []
        while len(pts) < T:
            p = torch.randint(lo, hi + 1, (2,), generator=g).float()
            pts += [p] * int(torch.randint(1, 5, (1,), generator=g))
        xy = torch.stack(pts[:T])[torch.randperm(T, generator=g)]
        pose[b] = torch.cat([xy, (torch.rand(T, 1, generator=g) * 2 - 1) * 3], -1)
    return pose, torch.rand(Bt, T, generator=g) < p_inv


def _int_sources(B, S, g, p_inv=0.1, lo=-45, hi=45):
    xy = torch.randint(lo, hi + 1, (B, S, 2), generator=g).float()
    return torch.cat([xy, torch.zeros(B, S, 1)], -1), torch.rand(B, S, generator=g) < p_inv


def _knn_expected(src, sinv, tgt, tinv, K, lim, div=1):
    """First K of a stable sort by (float64 distance, index), in ascending index order; invalid = target invalid or
    d > lim; relative pose in the (yaw 0) source frame."""
    tg, ti = tgt.double().repeat_interleave(div, 0), tinv.repeat_interleave(div, 0)
    dx = tg[:, None, :, 0] - src.double()[:, :, None, 0]
    dy = tg[:, None, :, 1] - src.double()[:, :, None, 1]
    d = (dx * dx + dy * dy).sqrt().masked_fill(sinv[:, :, None] | ti[:, None, :], math.inf)
    idx = torch.sort(d, dim=-1, stable=True)[1][..., :K].sort(-1)[0]
    dk = torch.gather(d, 2, idx)
    inv = torch.gather(ti[:, None].expand(-1, src.shape[1], -1), 2, idx) | (dk > lim)
    yaw = torch.gather(tg[:, None, :, 2].expand(-1, src.shape[1], -1), 2, idx)
    rel = torch.stack([torch.gather(dx, 2, idx), torch.gather(dy, 2, idx), yaw], -1).float()
    return idx.to(torch.int32), inv, rel


def _check_knn_exact(src, sinv, tgt, tinv, K, lim, div=1, what=""):
    dv = lambda t: t.contiguous().to(DEV)  # noqa: E731
    idx, inv, rel = ops.knn_select(dv(src), dv(sinv), dv(tgt), dv(tinv), K, lim, tgt_div=div)
    e_idx, e_inv, e_rel = _knn_expected(src, sinv, tgt, tinv, K, lim, div)
    idx, inv, rel = idx.cpu(), inv.cpu(), rel.cpu()
    bad = (idx != e_idx).any(-1)
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} rows differ, first {idx[bad][0].tolist()} vs {e_idx[bad][0].tolist()}"
    assert torch.equal(inv, e_inv), f"{what}: invalid flags"
    assert torch.equal(rel, e_rel), f"{what}: relative poses"


KNN_T = [33, 64, 65, 128, 129, 256, 257, 512, 513, 1024, 1025, 2048]


@pytest.mark.parametrize("T", KNN_T)
def test_knn_select_exact_ties(T):
    """Every targets-per-lane boundary, K in {1, 32, 33, 64, 65, T - 1}: full scan (T <= 128, K > 64) and prune path.
    Scene 1 has fewer valid targets than most K, some sources are invalid; dist_limit 25 has targets at exactly 25."""
    g = torch.Generator().manual_seed(T)
    B, S = 3, 40
    tgt, tinv = _grid_targets(B, T, g)
    tinv[1] = torch.rand(T, generator=g) < 0.97
    src, sinv = _int_sources(B, S, g)
    src[0, 0, :2] = torch.tensor([0.0, 0.0])
    sinv[0, 0] = False
    tgt[0, :4, :2] = torch.tensor([[15.0, 20.0], [-20.0, 15.0], [25.0, 0.0], [7.0, 24.0]])  # exactly 25 from src[0, 0]
    tinv[0, :4] = False
    for K in sorted({k for k in (1, 32, 33, 64, 65, T - 1) if k < T}):
        _check_knn_exact(src, sinv, tgt, tinv, K, 25.0, what=f"T={T} K={K}")


def test_knn_select_exact_ties_shared_tables():
    """Target tables shared by div = 3 consecutive source batches, and dist_limit 5 on 3-4-5 triangles."""
    g = torch.Generator().manual_seed(5)
    tgt, tinv = _grid_targets(2, 300, g, lo=-8, hi=8)
    src, sinv = _int_sources(6, 50, g, lo=-8, hi=8)
    for K in (5, 40, 64, 100):
        _check_knn_exact(src, sinv, tgt, tinv, K, 5.0, div=3, what=f"div=3 K={K}")


def _prune_survivors(src, sinv, tgt, tinv, K, div):
    """Keys at or below the prune bound of knn_select.cu:214-227 for every source row: U = max over the 32 lanes of the
    lane's smallest (K <= 32) or second-smallest key, lane l holding targets l, l + 32, ... Invalid targets rank
    above every distance, the padding of the last lane row above those."""
    T = tgt.shape[1]
    tpl = max(2, 1 << (T - 1).bit_length()) // 32
    tg, ti = tgt.double().repeat_interleave(div, 0), tinv.repeat_interleave(div, 0)
    dx = tg[:, None, :, 0] - src.double()[:, :, None, 0]
    dy = tg[:, None, :, 1] - src.double()[:, :, None, 1]
    key = (dx * dx + dy * dy).masked_fill(ti[:, None, :], 1e200)
    key = torch.cat([key, torch.full(key.shape[:2] + (tpl * 32 - T,), 1e300, dtype=key.dtype)], -1)
    lane_sorted = key.view(*key.shape[:2], tpl, 32).sort(2)[0]
    U = lane_sorted[:, :, 0 if K <= 32 else 1].amax(-1)
    return (key <= U[..., None]).sum(-1)[~sinv]


@pytest.mark.parametrize("T", [513, 1024, 2048])
def test_knn_select_prune_overflow(T):
    """More than kCap * 32 = 384 keys at or below the prune bound U: the prune path falls back to the bisection over
    all keys (knn_select.cu:227). (a) sources 400+ m from a 5 m target cloud, most of it stacked on its nearest point (an
    evenly spread cloud keeps ~20 % of the keys); (b) a ring: every valid target at distance exactly 5, so all keys
    tie and need_ties = K. The bound is recomputed here to show that every valid row takes the fallback."""
    g = torch.Generator().manual_seed(T + 1)
    B, S = 2, 24
    cloud, cinv = _grid_targets(1, T, g, p_inv=0.05, lo=100, hi=105)
    cloud[0, torch.rand(T, generator=g) < 0.9, :2] = 100.0  # the corner nearest to every source
    src, sinv = _int_sources(B, S, g, p_inv=0.1, lo=-400, hi=-300)
    ring_pts = torch.tensor([[5, 0], [-5, 0], [0, 5], [0, -5], [3, 4], [3, -4], [-3, 4], [-3, -4], [4, 3], [4, -3],
                             [-4, 3], [-4, -3]], dtype=torch.float32)
    ring = torch.cat([ring_pts[torch.randint(0, 12, (T,), generator=g)], torch.rand(T, 1, generator=g)], -1)[None]
    rinv = torch.rand(1, T, generator=g) < 0.1
    rsrc = torch.zeros(B, S, 3)
    rsinv = torch.zeros(B, S, dtype=torch.bool)
    for K in (1, 32, 33, 64):
        assert int(_prune_survivors(src, sinv, cloud, cinv, K, B).min()) > 384
        assert int(_prune_survivors(rsrc, rsinv, ring, rinv, K, B).min()) > 384
        _check_knn_exact(src, sinv, cloud, cinv, K, 1e9, div=B, what=f"cloud T={T} K={K}")
        _check_knn_exact(rsrc, rsinv, ring, rinv, K, 5.0, div=B, what=f"ring T={T} K={K}")


@pytest.mark.parametrize("K", [25, 64])
def test_knn_select_slab_path_exact_geometry(K):
    """x-sorted static targets + row_state (sorted_by_x): the tie choice among equal distances is free here (DESIGN
    §5), so check that the selected distances equal the K smallest as multisets, without duplicates, with consistent
    flags and exact relative poses, over a few moving steps."""
    B, S, T, lim = 2, 50, 1024, 20.0
    g = torch.Generator().manual_seed(K)
    tgt, tinv = _grid_targets(1, T, g)
    order = torch.argsort(tgt[..., 0], dim=1, stable=True)
    s_pose = torch.gather(tgt, 1, order[..., None].expand(-1, -1, 3)).contiguous()
    s_inv = torch.gather(tinv, 1, order).contiguous()
    state = torch.full((B, S, 3), float("inf"), device=DEV)
    src, _ = _int_sources(B, S, g)
    armed = False
    for step in range(5):
        sinv = torch.rand(B, S, generator=g) < 0.1
        if step:
            src[..., :2] += torch.randint(-3, 4, (B, S, 2), generator=g).float()
        idx, inv, rel = ops.knn_select(src.to(DEV), sinv.to(DEV), s_pose.to(DEV), s_inv.to(DEV), K, lim, tgt_div=B,
                                       index_map=order.to(torch.int32).contiguous().to(DEV), row_state=state,
                                       sorted_by_x=True)
        idx, inv, rel = idx.cpu().long(), inv.cpu(), rel.cpu()
        _, e_inv, _ = _knn_expected(src, sinv, tgt, tinv, K, lim, div=B)
        tg, ti = tgt.double().expand(B, -1, -1), tinv.expand(B, -1)
        dx = tg[:, None, :, 0] - src.double()[:, :, None, 0]
        dy = tg[:, None, :, 1] - src.double()[:, :, None, 1]
        d = (dx * dx + dy * dy).sqrt().masked_fill(sinv[:, :, None] | ti[:, None, :], math.inf)
        ok = ~sinv
        assert bool((idx.sort(-1)[0][..., 1:] > idx.sort(-1)[0][..., :-1]).all()), f"step {step}: duplicates"
        sel = torch.gather(d, 2, idx).sort(-1)[0]
        assert torch.equal(sel[ok], d.sort(-1)[0][..., :K][ok]), f"step {step}: distances are not the K smallest"
        exp_inv = torch.gather(ti[:, None].expand(-1, S, -1), 2, idx) | (torch.gather(d, 2, idx) > lim)
        assert torch.equal(inv, exp_inv), f"step {step}: invalid flags"
        assert torch.equal(inv.sum(-1)[ok], e_inv.sum(-1)[ok])
        exp_rel = torch.stack([torch.gather(dx, 2, idx), torch.gather(dy, 2, idx),
                               torch.gather(tg[:, None, :, 2].expand(-1, S, -1), 2, idx)], -1).float()
        assert torch.equal(rel[ok], exp_rel[ok]), f"step {step}: relative poses"
        armed = armed or bool(torch.isfinite(state[..., 2]).any())
    assert armed


def test_knn_select_grid_limit():
    """One CTA row per source batch in the grid's y dimension: B = 65535 runs (checked), B = 65536 is refused."""
    g = torch.Generator().manual_seed(3)
    T, K = 33, 1
    tgt, tinv = _grid_targets(1, T, g, p_inv=0.0)
    B = 65535
    src, sinv = _int_sources(B, 1, g)
    _check_knn_exact(src, sinv, tgt, tinv, K, 30.0, div=B, what="B=65535")
    src2 = torch.zeros(B + 1, 1, 3, device=DEV)
    with pytest.raises(RuntimeError, match="unsupported"):
        ops.knn_select(src2, torch.zeros(B + 1, 1, dtype=torch.bool, device=DEV), tgt.to(DEV), tinv.to(DEV), K, 30.0,
                       tgt_div=B + 1)
