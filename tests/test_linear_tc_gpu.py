"""GPU: the tensor-core projection kernel (linear_tc.cu: tb_linear precision 1 / 2, tb_linear_ln) branch by branch
against the float64 references of tests/_linear_ref.py.

(a) Accumulator: no bias or epilogue, against sum x~ w~ over the operands the tensor core multiplies, within the
    derived accumulation bound; every run bit-identical to a repeat and to the same call on a strided X view.
(b) Epilogue: every bias / ReLU / mask / residual variant bit-identical to the fp32 epilogue applied to (a)'s
    accumulator, on the vector store path (aligned views) and on the scalar one (N tails, views offset by one float
    with ld % 4 != 0).
(c) fp16 outputs: Yh bit-identical to the satfinite rounding of the fp32 result, on 8- and 2-byte aligned views; the
    fp16 range flag set exactly when a Yh value reaches 65504.
(d) Fused LayerNorm: Y bit-identical to tb_linear's, ln_out within the derived bound of LayerNorm(Y) in float64 at
    row mean / std up to 1000, masked rows exactly fp16(beta).
Unused memory around every output is sentinel-filled and must come back unchanged; memory past K / M / N in the
operands is NaN and must not reach the output. The projection forms a default-options rollout issues are recorded
and must all be in this file's case tables."""
import math
import zlib

import pytest
import torch

import _linear_ref as LR
from trafficbotsv1_5_b200 import config, params, synth

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from trafficbotsv1_5_b200 import ops

DEV = "cuda"
S32, S16 = 0x7FBADBAD, 0x7E5A  # NaN bit patterns of never-written memory
BIG = 3 * 148 * 128 + 77        # more than two 128-row tiles per CTA for any N on 148 SMs
WORST = {1: 0.0, 2: 0.0, "ln": 0.0}

# (a) accumulator shapes: every M, N and K of the sweep appears; (M, N, K)
ACC_CASES = {
    1: [(1, 2, 4), (127, 5, 20), (128, 6, 36), (129, 17, 100), (4097, 40, 128), (BIG, 64, 132), (129, 121, 640),
        (4097, 128, 1920), (127, 129, 36), (1, 200, 128), (BIG, 200, 20), (4097, 896, 128), (128, 896, 1920),
        (BIG, 17, 640), (128, 64, 4), (129, 2, 1920)],
    2: [(1, 2, 8), (127, 5, 24), (128, 6, 72), (129, 17, 136), (4097, 40, 512), (BIG, 64, 24), (129, 121, 512),
        (4097, 128, 136), (127, 129, 8), (1, 200, 72), (BIG, 200, 136), (4097, 896, 512), (128, 896, 8),
        (BIG, 6, 72)],
}
# (b) epilogue shapes: (precision, M, N, K)
EPI_CASES = [(1, 4097, 128, 128), (1, 129, 200, 36), (1, BIG, 40, 20), (2, 1000, 896, 136), (2, 300, 17, 24),
             (1, 1, 64, 100), (1, 2000, 5, 384)]
# (c) fp16 outputs: (precision, M, N, K, col_h)
F16_CASES = [(1, 1000, 896, 128, 640), (1, 300, 200, 36, 96), (2, 129, 129, 24, 32), (1, 4097, 64, 20, 0),
             (2, 1000, 121, 72, 96), (2, BIG, 256, 136, 0), (1, 2000, 768, 128, 0)]
# (d) fused LayerNorm: (precision, M, K, extras) with m = mask_pre, r = residual, p = mask_post
LN_CASES = [(2, 4097, 640, "mr"), (1, 1000, 128, "rp"), (2, 77, 512, ""), (1, BIG, 132, "mrp"), (2, 300, 128, "p"),
            (2, 1000, 512, "rp")]
# Projection forms of a default-options rollout (test_engine_projection_forms_are_covered):
# (precision, N, K, bias kind, relu, mask_pre, residual, mask_post, col_h or None without Yh); fused LayerNorm forms
# as ("ln", precision, N, K, bias kind, mask_pre, residual, mask_post).
# Forms with K % 4 != 0 run the fp32 FFMA kernel (no TMA rows) and are checked as that fallback.
ENGINE_FORMS = {
    ("ln", 2, 128, 512, "plain", False, True, True), ("ln", 2, 128, 640, "plain", True, True, False),
    (1, 121, 121, "plain", False, False, False, False, None), (1, 121, 121, "plain", True, False, False, False, None),
    (1, 121, 31, "plain", True, False, False, False, None), (1, 128, 128, "plain", False, False, False, False, None),
    (1, 128, 128, "plain", False, False, True, False, None), (1, 128, 128, "plain", True, False, False, False, None),
    (1, 128, 128, "plain", True, False, False, True, None), (1, 128, 16, "plain", True, False, False, False, None),
    (1, 5, 128, "plain", False, False, False, False, None), (1, 64, 128, "plain", True, False, False, False, None),
    (1, 64, 64, "group", True, False, False, False, None), (1, 64, 64, "plain", False, False, False, False, None),
    (2, 128, 512, "plain", False, False, True, True, None), (2, 256, 128, "plain", False, False, False, False, 0),
    (2, 512, 128, "plain", True, False, False, False, 0), (2, 640, 128, "plain", False, False, False, False, 0),
    (2, 896, 128, "plain", False, False, False, False, 0),
}


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


class Buf:
    """A rows x cols view with leading dim ld at element offset `off` inside a sentinel-filled flat buffer with extra
    rows after it; `untouched()` checks every element outside the view."""

    def __init__(self, rows, cols, ld, off=0, dtype=torch.float32, fill=None):
        n = off + (rows + 2) * ld + 8
        self.buf = torch.empty(n, dtype=dtype, device=DEV)
        _bits(self.buf).fill_(S32 if dtype == torch.float32 else S16)
        self.view = self.buf[off:off + rows * ld].view(rows, ld)[:, :cols]
        if fill is not None:
            self.view.copy_(fill)
        self.mask = torch.zeros(n, dtype=torch.bool, device=DEV)
        self.mask[off:off + rows * ld].view(rows, ld)[:, :cols] = True
        self.sentinel = S32 if dtype == torch.float32 else S16

    def untouched(self):
        return bool((_bits(self.buf)[~self.mask] == self.sentinel).all())


def _operand(rows, cols, ld, prec, g, scale=1.0, off=0):
    """rows x cols values in a NaN-filled buffer: row padding past `cols` and 3 rows past `rows` are NaN."""
    dt = torch.float16 if prec == 2 else torch.float32
    buf = torch.full((off + (rows + 3) * ld,), float("nan"), dtype=dt, device=DEV)
    v = buf[off:off + rows * ld].view(rows, ld)[:, :cols]
    v.copy_((torch.randn(rows, cols, generator=g, device=DEV) * scale).to(dt))
    return v


def _weight(N, K, prec, g):
    """[N, K] contiguous weights (1/sqrt(K) scale) followed in memory by 5 NaN rows."""
    dt = torch.float16 if prec == 2 else torch.float32
    buf = torch.full(((N + 5) * K,), float("nan"), dtype=dt, device=DEV)
    w = buf[:N * K].view(N, K)
    w.copy_((torch.randn(N, K, generator=g, device=DEV) / math.sqrt(K)).to(dt))
    return w


def _ld(n, vector):
    """A leading dim >= n: a multiple of 4 (vector store path) or 1 mod 4 (scalar path)."""
    return (n + 3) // 4 * 4 + (4 if vector else 5)


def _acc(x, w, prec):
    """The kernel's accumulator (no bias, no epilogue) as a contiguous [M, N] fp32 tensor."""
    return ops.linear(x, w, None, precision=prec)


# ------------------------------------------------------------------------------------------------ (a) accumulator
@pytest.mark.parametrize("prec,M,N,K", [(p,) + c for p in (1, 2) for c in ACC_CASES[p]])
def test_accumulator_within_bound_and_deterministic(prec, M, N, K):
    g = _gen(M * 7 + N * 3 + K + prec)
    ldx = K + (12 if prec == 1 else 8)  # strided X rows (TMA needs 16-byte rows); the padding is NaN
    x, w = _operand(M, K, ldx, prec, g), _weight(N, K, prec, g)
    outs = []
    for _ in range(2):
        o = Buf(M, N, _ld(N, True))
        ops.linear(x, w, None, out=o.view, precision=prec)
        outs.append(o)
    dense = ops.linear(x.contiguous(), w, None, precision=prec)
    torch.cuda.synchronize()
    y = outs[0].view
    assert bool(torch.isfinite(y).all()), "NaN padding of X / W reached the output"
    assert all(o.untouched() for o in outs), "written outside the output view"
    assert torch.equal(_bits(y), _bits(outs[1].view)), "repeat run differs"
    assert torch.equal(_bits(y), _bits(dense)), "strided X differs from contiguous X"
    err = (y.double() - LR.acc_ref(x, w, prec)).abs()
    bound = LR.acc_bound(x, w, prec)
    r = float((err / bound.clamp_min(1e-300)).max())
    WORST[prec] = max(WORST[prec], r)
    print(f"\naccumulator p{prec} {M}x{N}x{K}: worst error / bound {r:.3g} (all cases so far: {WORST[prec]:.3g})")
    assert r <= 1.0, f"{int((err > bound).sum())} elements outside the accumulation bound, worst {r:.3g} x"


# ------------------------------------------------------------------------------------------------ (b) epilogue
def _divisor(M):
    return next((d for d in range(2, 64) if M % d == 0), M)


def _epi_inputs(M, N, g, bias, vector):
    """(bias tensor, group, res view, mask_pre, mask_post) for one variant, on aligned views (vector) or views
    offset by one float with ld % 4 != 0 (scalar path)."""
    off = 0 if vector else 1
    grp = 0
    b = None
    if bias is not None:
        grp = bias
        rows = (M + grp - 1) // grp if grp else 1
        flat = torch.empty(off + rows * N, device=DEV)
        flat[off:] = torch.randn(rows * N, generator=g, device=DEV)  # the same values on both paths
        b = flat[off:].view(rows, N) if grp else flat[off:]
    ldr = _ld(N, vector)
    res = Buf(M, N, ldr, off, fill=torch.randn(M, N, generator=g, device=DEV) * 0.5).view
    mpre = torch.rand(M, generator=g, device=DEV) < 0.3
    mpost = torch.rand(M, generator=g, device=DEV) < 0.3
    return b, grp, res, mpre, mpost


def _variants(M):
    """bias kinds: None, plain (0), grouped by a divisor of M and by a non-divisor; x ReLU x the 8 row-extra sets."""
    nd = next(d for d in range(3, 64) if M % d)
    for bias in (None, 0, _divisor(M), nd):
        for relu in (False, True):
            for ex in range(8):
                yield bias, relu, bool(ex & 1), bool(ex & 2), bool(ex & 4)


@pytest.mark.parametrize("prec,M,N,K", EPI_CASES)
def test_epilogue_bit_exact_on_both_store_paths(prec, M, N, K):
    g = _gen(M + N + K)
    x, w = _operand(M, K, K, prec, g), _weight(N, K, prec, g)
    acc = _acc(x, w, prec)
    n = 0
    for bias, relu, use_pre, use_res, use_post in _variants(M):
        got = {}
        for vector in (True, False):
            b, grp, res, mpre, mpost = _epi_inputs(M, N, _gen(n), bias, vector)
            kw = dict(relu=relu, mask_pre=mpre if use_pre else None, res=res if use_res else None,
                      mask_post=mpost if use_post else None)
            o = Buf(M, N, _ld(N, vector), 0 if vector else 1)
            ops.linear(x, w, b, out=o.view, precision=prec, bias_group=grp, **kw)
            ref = LR.epilogue_f32(acc, b, grp, **kw)
            what = f"bias {bias} relu {relu} pre {use_pre} res {use_res} post {use_post} {'vector' if vector else 'scalar'}"
            assert LR.same_bits(o.view, ref), f"{what}: {int((o.view != ref).sum())} elements differ from the fp32 epilogue"
            assert o.untouched(), f"{what}: written outside the output view"
            got[vector] = o.view
        assert LR.same_bits(got[True], got[False])
        n += 1
    assert n == 64


# ------------------------------------------------------------------------------------------------ (c) fp16 outputs
@pytest.mark.parametrize("prec,M,N,K,col_h", F16_CASES)
def test_fp16_output_is_satfinite_of_fp32_result(prec, M, N, K, col_h):
    g = _gen(M + N + K + col_h)
    x, w = _operand(M, K, K, prec, g), _weight(N, K, prec, g)
    b = torch.randn(N, generator=g, device=DEV)
    mpre, mpost = torch.rand(M, generator=g, device=DEV) < 0.3, torch.rand(M, generator=g, device=DEV) < 0.3
    res = torch.randn(M, N, generator=g, device=DEV)
    flag = ops.fp16_flag(DEV)
    for extras in ({}, dict(relu=True, mask_pre=mpre, res=res, mask_post=mpost), dict(res=res, mask_post=mpost)):
        full = ops.linear(x, w, b, precision=prec, **extras)
        for vector in (True, False):
            hb = Buf(M, N - col_h, _ld(N - col_h, vector), 0 if vector else 1, dtype=torch.float16)
            yb = Buf(M, N, _ld(N, True)) if col_h else None  # columns >= col_h of the fp32 rows stay sentinel
            flag.zero_()
            r = ops.linear(x, w, b, out=yb.view[:, :col_h] if col_h else None, precision=prec, out_h=hb.view,
                           col_h=col_h, **extras)
            torch.cuda.synchronize()
            what = f"{sorted(extras)} {'8-byte' if vector else '2-byte'} Yh"
            assert LR.same_bits(hb.view, LR.sat_f16(full[:, col_h:])), f"{what}: Yh is not satfinite(fp32 result)"
            assert hb.untouched(), f"{what}: Yh written outside its view"
            if col_h:
                assert r.data_ptr() == yb.view.data_ptr()
                assert torch.equal(_bits(yb.view[:, :col_h]), _bits(full[:, :col_h])), what
                assert yb.untouched() and bool((_bits(yb.view[:, col_h:]) == S32).all()), \
                    f"{what}: fp32 rows written at columns >= col_h"
            else:
                assert r is None
            assert int(flag.item()) == int(bool((LR.sat_f16(full[:, col_h:]).abs() == LR.F16_MAX).any())), what


@pytest.mark.parametrize("where", ["vector", "tail", "misaligned"])
def test_fp16_range_flag(where):
    """The sticky fp16 range flag: set when a Yh value reaches +-65504 (vector store path, the scalar N tail, a
    2-byte-aligned Yh), clear when every Yh value is below it even though an fp32 column (< col_h) is far above."""
    M, N, K, col_h = 300, 200, 64, 96
    g = _gen(41)
    x, w = _operand(M, K, K, 1, g, scale=0.1), _weight(N, K, 1, g)
    flag = ops.fp16_flag(DEV)
    hot = {"vector": col_h + 7, "tail": 197, "misaligned": col_h + 7}[where]
    vector = where != "misaligned"
    for big_col, value, expect in ((5, 1e6, 0), (hot, 6.0e4, 0), (hot, -7.0e4, 1), (hot, 65504.0, 1)):
        b = torch.zeros(N, device=DEV)
        b[big_col] = value
        full = ops.linear(x, w, b, precision=1)
        hb = Buf(M, N - col_h, _ld(N - col_h, vector), 0 if vector else 1, dtype=torch.float16)
        y = torch.empty(M, col_h, device=DEV)
        flag.zero_()
        ops.linear(x, w, b, out=y, precision=1, out_h=hb.view, col_h=col_h)
        torch.cuda.synchronize()
        assert int(flag.item()) == expect, (where, big_col, value)
        assert LR.same_bits(hb.view, LR.sat_f16(full[:, col_h:])) and hb.untouched()
        if expect:
            assert bool((hb.view[:, hot - col_h].float().abs() == LR.F16_MAX).all())


# ------------------------------------------------------------------------------------------------ (d) fused LayerNorm
def _ln_inputs(prec, M, K, g, offsets=None):
    x, w = _operand(M, K, K, prec, g), _weight(128, K, prec, g)
    b = torch.randn(128, generator=g, device=DEV) * 0.1
    gamma, beta = torch.rand(128, generator=g, device=DEV) + 0.5, torch.randn(128, generator=g, device=DEV)
    res = torch.randn(M, 128, generator=g, device=DEV) * 0.5
    if offsets is not None:
        res += offsets[:, None]
    return x, w, b, gamma, beta, res


def _check_ln(prec, M, x, w, b, gamma, beta, kw, what):
    y0 = ops.linear(x, w, b, precision=prec, **kw)
    y, ln = ops.linear_ln(x, w, b, gamma, beta, precision=prec, **kw)
    torch.cuda.synchronize()
    assert torch.equal(_bits(y), _bits(y0)), f"{what}: Y differs from tb_linear's"
    ref, mu, var = LR.layernorm_ref_f64(y, gamma, beta)
    bound = LR.ln_out_bound(y, gamma, beta)
    err = (ln.double() - ref).abs()
    r = float((err / bound).max())
    WORST["ln"] = max(WORST["ln"], r)
    if kw.get("mask_post") is not None:
        mp = kw["mask_post"]
        assert torch.equal(_bits(ln[mp]), _bits(beta.half().expand(int(mp.sum()), 128))), f"{what}: masked rows"
    assert r <= 1.0, f"{what}: {int((err > bound).sum())} ln_out values outside the bound, worst {r:.3g} x"
    return r, float((mu.abs() / var.sqrt().clamp_min(1e-30)).max())


@pytest.mark.parametrize("prec,M,K,extras", LN_CASES)
def test_fused_layernorm(prec, M, K, extras):
    g = _gen(M + K)
    x, w, b, gamma, beta, res = _ln_inputs(prec, M, K, g)
    kw = dict(mask_pre=(torch.rand(M, generator=g, device=DEV) < 0.2) if "m" in extras else None,
              res=res if "r" in extras else None,
              mask_post=(torch.rand(M, generator=g, device=DEV) < 0.2) if "p" in extras else None)
    _check_ln(prec, M, x, w, b, gamma, beta, kw, f"p{prec} {M}x{K} {extras}")


@pytest.mark.parametrize("ratio", [0, 10, 100, 1000])
@pytest.mark.parametrize("prec", [1, 2])
def test_fused_layernorm_rows_far_from_zero(prec, ratio):
    """Rows whose mean is `ratio` times their spread (the residual adds a per-row offset, the GEMM part keeps the
    spread O(1)): the statistics must not lose the variance to cancellation."""
    M, K = 2 * 148 * 128 + 33, 128
    g = _gen(ratio + prec)
    off = ratio * (1.0 + 0.1 * torch.rand(M, generator=g, device=DEV)) * torch.where(
        torch.rand(M, generator=g, device=DEV) < 0.5, -1.0, 1.0)
    x, w, b, gamma, beta, res = _ln_inputs(prec, M, K, g, off)
    mpost = torch.rand(M, generator=g, device=DEV) < 0.05
    r, mr = _check_ln(prec, M, x, w, b, gamma, beta, dict(res=res, mask_post=mpost), f"p{prec} mean/std ~ {ratio}")
    print(f"\nfused LayerNorm p{prec} mean/std up to {mr:.0f}: worst ln_out error / bound {r:.3g}")


# ------------------------------------------------------------------------------------------------ fallbacks, refusals
@pytest.mark.parametrize("form", ["k_mod4", "ldx_mod4", "x_misaligned"])
def test_shapes_outside_tma_fall_back_or_refuse(form):
    """Precision 1 on shapes the TMA path cannot take runs the fp32 FFMA kernel: bit-identical to precision 0. With a
    Yh output or fp16 operands those shapes are refused and the outputs stay untouched."""
    M, N = 1000, 96
    K = {"k_mod4": 18, "ldx_mod4": 64, "x_misaligned": 64}[form]
    ldx = {"k_mod4": 18, "ldx_mod4": 66, "x_misaligned": 64}[form]
    g = _gen(7)
    x = _operand(M, K, ldx, 1, g, off=1 if form == "x_misaligned" else 0)
    w = _weight(N, K, 1, g)
    b, res = torch.randn(N, generator=g, device=DEV), torch.randn(M, N, generator=g, device=DEV)
    mp = torch.rand(M, generator=g, device=DEV) < 0.3
    kw = dict(relu=True, mask_pre=mp, res=res, mask_post=~mp)
    y1, y0 = ops.linear(x, w, b, precision=1, **kw), ops.linear(x, w, b, precision=0, **kw)
    assert torch.equal(_bits(y1), _bits(y0))
    yb, hb = Buf(M, 32, 36), Buf(M, N - 32, N - 28, dtype=torch.float16)
    with pytest.raises(RuntimeError):
        ops.linear(x, w, b, out=yb.view, precision=1, out_h=hb.view, col_h=32, **kw)
    x16 = _operand(M, K, ldx + (2 if form == "ldx_mod4" else 0), 2, g, off=1 if form == "x_misaligned" else 0)
    yf = Buf(M, N, N + 4)
    with pytest.raises(RuntimeError):  # K % 8, ldx % 8 (68) or a 2-byte-aligned X: no fp16 FFMA kernel
        ops.linear(x16, _weight(N, K, 2, g), b, out=yf.view, precision=2)
    torch.cuda.synchronize()
    for o in (yb, hb, yf):
        assert o.untouched() and bool((_bits(o.view) == o.sentinel).all()), "a refused call wrote its outputs"


# ------------------------------------------------------------------------------------------------ engine coverage
def _bias_kind(b, grp):
    return "none" if b is None else ("group" if grp else "plain")


def test_engine_projection_forms_are_covered(monkeypatch):
    """Every (precision, N, K, bias kind, ReLU, masks, residual, col_h) form that a default-options tensor-core rollout
    sends to linear_tc must be one this file checks (ENGINE_FORMS, run by test_engine_forms_bit_exact): a projection
    form the engine adds later fails here until it is covered."""
    from trafficbotsv1_5_b200.engine import RolloutEngine
    seen = set()
    lin, lin_ln = ops.linear, ops.linear_ln

    def rec_linear(x, w, b=None, relu=False, mask_pre=None, res=None, mask_post=None, out=None, precision=0,
                   bias_group=0, out_h=None, col_h=0):
        if precision in (1, 2):
            seen.add((precision, w.shape[0], w.shape[1], _bias_kind(b, bias_group), bool(relu), mask_pre is not None,
                      res is not None, mask_post is not None, col_h if out_h is not None else None))
        return lin(x, w, b, relu, mask_pre, res, mask_post, out, precision, bias_group, out_h, col_h)

    def rec_linear_ln(x, w, b, gamma, beta, mask_pre=None, res=None, mask_post=None, out=None, precision=2):
        seen.add(("ln", precision, w.shape[0], w.shape[1], _bias_kind(b, 0), mask_pre is not None, res is not None,
                  mask_post is not None))
        return lin_ln(x, w, b, gamma, beta, mask_pre, res, mask_post, out, precision)

    monkeypatch.setattr(ops, "linear", rec_linear)
    monkeypatch.setattr(ops, "linear_ln", rec_linear_ln)
    cfg = config.default_model_cfg()
    P = params.init_params(cfg, 0)
    batch = synth.make_scene_batch(n_sc=2, n_ag=32, n_mp=96, n_tl=30, seed=11, boundary=105.0)
    eng = RolloutEngine(P, cfg, DEV, precision=1, n_rollout=2, step_end=14)
    eng.rollout(batch)
    torch.cuda.synchronize()
    assert seen, "no projection reached linear_tc"
    missing = sorted(seen - ENGINE_FORMS, key=str)
    assert not missing, f"projection forms not covered by ENGINE_FORMS: {missing}"


@pytest.mark.parametrize("form", sorted(ENGINE_FORMS, key=str))
def test_engine_forms_bit_exact(form):
    """Each engine projection form at a partial row block: the accumulator within its bound, the epilogue bit-exact,
    Yh the satfinite rounding of the fp32 result, the fused LayerNorm within its bound."""
    M = 1000
    g = _gen(zlib.crc32(str(form).encode()))
    if form[0] == "ln":
        _, prec, N, K, bk, pre, rs, post = form
        x, w, b, gamma, beta, res = _ln_inputs(prec, M, K, g)
        kw = dict(mask_pre=(torch.rand(M, generator=g, device=DEV) < 0.2) if pre else None, res=res if rs else None,
                  mask_post=(torch.rand(M, generator=g, device=DEV) < 0.2) if post else None)
        _check_ln(prec, M, x, w, None if bk == "none" else b, gamma, beta, kw, str(form))
        return
    prec, N, K, bk, relu, pre, rs, post, col_h = form
    x, w = _operand(M, K, K, prec, g), _weight(N, K, prec, g)
    grp = 16 if bk == "group" else 0
    b = None if bk == "none" else torch.randn(((M + grp - 1) // grp, N) if grp else (N,), generator=g, device=DEV)
    kw = dict(relu=relu, mask_pre=(torch.rand(M, generator=g, device=DEV) < 0.3) if pre else None,
              res=torch.randn(M, N, generator=g, device=DEV) if rs else None,
              mask_post=(torch.rand(M, generator=g, device=DEV) < 0.3) if post else None)
    if K % 4:
        assert prec == 1 and col_h is None
        y1, y0 = (ops.linear(x, w, b, precision=p, bias_group=grp, **kw) for p in (1, 0))
        assert torch.equal(_bits(y1), _bits(y0)), "K % 4 must run the FFMA kernel"
        return
    acc = _acc(x, w, prec)
    err = (acc.double() - LR.acc_ref(x, w, prec)).abs()
    assert bool((err <= LR.acc_bound(x, w, prec)).all())
    ref = LR.epilogue_f32(acc, b, grp, **kw)
    if col_h is None:
        assert LR.same_bits(ops.linear(x, w, b, precision=prec, bias_group=grp, **kw), ref)
    else:
        yh = torch.empty(M, N - col_h, dtype=torch.float16, device=DEV)
        y = ops.linear(x, w, b, precision=prec, bias_group=grp, out_h=yh, col_h=col_h, **kw)
        assert LR.same_bits(yh, LR.sat_f16(ref[:, col_h:]))
        if col_h:
            assert LR.same_bits(y, ref[:, :col_h])
