"""CPU: the float64 reference helpers of the projection tests (tests/_linear_ref.py) and every argument refusal of
tb_linear / tb_linear_ln. The refusals are returned by api.cu and the top of tb_linear_tc before any CUDA call, so they
are checked with fake device addresses (never dereferenced) and no device."""
import pytest
import torch

import _linear_ref as LR
from trafficbotsv1_5_b200 import lib

TB_ERR_BAD_SHAPE, TB_ERR_UNSUPPORTED, TB_ERR_MISALIGNED, TB_ERR_NULL = -1, -3, -4, -5
A = 1 << 20  # fake 16-byte-aligned device addresses: A, 2A, 3A, ...


@pytest.fixture(scope="module")
def handle():
    lib.build()
    return lib.load()


def test_trunc_tf32_keeps_sign_exponent_and_ten_mantissa_bits():
    x = torch.tensor([1.0, 1.0 + 2 ** -10, 1.0 + 2 ** -11, 1.0 + 2 ** -10 + 2 ** -11 + 2 ** -23, -3.999999, 2 ** -130,
                      65519.99, float("inf"), -0.0])
    t = LR.trunc_tf32(x)
    assert t.tolist()[:5] == [1.0, 1.0 + 2 ** -10, 1.0, 1.0 + 2 ** -10, -(2.0 - 2 ** -10) * 2]
    bits = t.view(torch.int32)
    assert bool(((bits & 8191) == 0).all())                                            # low 13 mantissa bits cleared
    assert torch.equal(bits >> 13, x.view(torch.int32) >> 13)                          # everything above them kept
    assert float(t[7]) == float("inf") and str(float(t[8])) == "-0.0"
    g = torch.Generator().manual_seed(1)
    r = torch.randn(10000, generator=g) * 10.0 ** torch.randint(-6, 6, (10000,), generator=g)
    rel = ((r.double() - LR.trunc_tf32(r).double()) / r.double()).abs()
    assert float(rel.max()) < 2 ** -10 and bool((LR.trunc_tf32(r).abs() <= r.abs()).all())  # toward zero, < 1 ulp


def test_sat_f16_is_round_to_nearest_with_saturation():
    x = torch.tensor([65504.0, 65519.99, 65520.0, 1e9, float("inf"), -65520.0, float("-inf"), 1.0 + 2 ** -11,
                      1.0 + 3 * 2 ** -11, 2 ** -25, 2 ** -25 * 3])
    h = LR.sat_f16(x).float().tolist()
    assert h[:7] == [65504.0, 65504.0, 65504.0, 65504.0, 65504.0, -65504.0, -65504.0]
    assert h[7] == 1.0 and h[8] == 1.0 + 2 ** -9                                       # ties to even
    assert h[9] == 0.0 and h[10] == 2 ** -23                                           # subnormal ties to even
    assert float(x[2].half()) == float("inf")                                          # plain rounding would overflow


def test_accumulator_reference_and_bound():
    g = torch.Generator().manual_seed(2)
    x, w = torch.randn(5, 20, generator=g), torch.randn(3, 20, generator=g)
    ref = LR.acc_ref(x, w, 1)
    assert torch.equal(ref, LR.trunc_tf32(x).double() @ LR.trunc_tf32(w).double().T)
    # products of tf32 / fp16 operands are exact in fp32 (at most 22 significant bits)
    p = LR.trunc_tf32(x)[:, None, :] * LR.trunc_tf32(w)[None, :, :]
    assert torch.equal(p.double(), LR.trunc_tf32(x).double()[:, None, :] * LR.trunc_tf32(w).double()[None, :, :])
    assert LR.gamma_acc(20, 1) == 5 * 2.0 ** -22 and LR.gamma_acc(16, 2) == 3 * 2.0 ** -22
    b = LR.acc_bound(x, w, 1)
    assert torch.allclose(b, LR.gamma_acc(20, 1) * (LR.trunc_tf32(x).double().abs() @ LR.trunc_tf32(w).double().abs().T))
    xh, wh = x.half(), w.half()
    assert torch.equal(LR.acc_ref(xh, wh, 2), xh.double() @ wh.double().T)
    # a plain fp32 sum of the same products lies inside the bound; the unrounded operands do not
    assert bool(((LR.trunc_tf32(x) @ LR.trunc_tf32(w).T).double() - ref).abs().le(b).all())
    assert not bool(((x @ w.T).double() - ref).abs().le(b).all())


def test_epilogue_reference_order():
    acc = torch.tensor([[1.0, -2.0, 3.0], [-4.0, 5.0, -6.0], [7.0, -8.0, 9.0]])
    b = torch.tensor([0.5, 0.5, -10.0])
    res = torch.full((3, 3), 100.0)
    mpre, mpost = torch.tensor([True, False, False]), torch.tensor([False, False, True])
    out = LR.epilogue_f32(acc, b, 0, True, mpre, res, mpost)
    assert out.tolist() == [[100.0, 100.0, 100.0], [100.0, 105.5, 100.0], [0.0, 0.0, 0.0]]
    gb = torch.tensor([[1.0, 1.0, 1.0], [2.0, 2.0, 2.0]])
    assert LR.epilogue_f32(acc, gb, 2).tolist() == (acc + torch.tensor([[1.0], [1.0], [2.0]])).tolist()
    # fp32 steps: (a + b) + r rounds twice
    a1 = torch.tensor([[1.0]]); r1 = torch.tensor([[2.0 ** -24]])
    assert float(LR.epilogue_f32(a1, torch.tensor([2.0 ** -24]), res=r1)) == 1.0


@pytest.mark.parametrize("ratio", [0, 10, 100, 1000])
def test_ln_bound_accepts_merged_statistics_and_rejects_one_pass(ratio):
    """ln_out_bound against fp32 emulations of the fused LayerNorm in the kernel's reduction order: the (sum, M2)
    partials merged with Chan's formula stay inside at every mean / std, the one-pass E[y^2] - E[y]^2 falls outside
    from mean / std = 100 (the rows tb_linear_ln has to get right once the residual stream drifts from zero)."""
    g = torch.Generator().manual_seed(ratio + 3)
    M = 512
    gamma, beta = torch.rand(128, generator=g) + 0.5, torch.randn(128, generator=g)
    y = torch.randn(M, 128, generator=g) * (0.5 + torch.rand(M, 1, generator=g))
    y = (y + ratio * y.std(1, keepdim=True)).float()
    ref, _, _ = LR.layernorm_ref_f64(y, gamma, beta)
    bd = LR.ln_out_bound(y, gamma, beta)
    merged = float(((LR.fused_ln_f32(y, gamma, beta).double() - ref).abs() / bd).max())
    one_pass = float(((LR.fused_ln_f32(y, gamma, beta, one_pass=True).double() - ref).abs() / bd).max())
    assert merged <= 1.0, merged
    assert (one_pass > 1.0) == (ratio >= 100), one_pass


def _lin(h, X=A, ldx=128, W=2 * A, bias=3 * A, bg=0, Y=4 * A, ldy=128, M=256, N=128, K=128, relu=0, mpre=None,
         res=None, ldr=0, mpost=None, prec=1, Yh=None, ldyh=0, col_h=0):
    return h.tb_linear(X, ldx, W, bias, bg, Y, ldy, M, N, K, relu, mpre, res, ldr, mpost, prec, Yh, ldyh, col_h, None)


def _ln(h, X=A, ldx=128, W=2 * A, bias=3 * A, Y=4 * A, ldy=128, M=256, N=128, K=128, mpre=None, res=None, ldr=0,
        mpost=None, prec=2, g=5 * A, b=6 * A, out=7 * A, ld_ln=128):
    return h.tb_linear_ln(X, ldx, W, bias, Y, ldy, M, N, K, mpre, res, ldr, mpost, prec, g, b, out, ld_ln, None)


def test_linear_refusals_without_gpu(handle):
    h = handle
    assert _lin(h, X=None) == TB_ERR_NULL and _lin(h, W=None) == TB_ERR_NULL
    for kw in (dict(M=0), dict(N=0), dict(K=0), dict(M=-1), dict(N=-5), dict(K=-8)):
        assert _lin(h, **kw) == TB_ERR_BAD_SHAPE, kw
    assert _lin(h, ldx=127) == TB_ERR_BAD_SHAPE                                      # ldx < K
    assert _lin(h, res=8 * A, ldr=127) == TB_ERR_BAD_SHAPE                           # ldr < N
    assert _lin(h, bg=-1) == TB_ERR_BAD_SHAPE
    yh = dict(Yh=8 * A, ldyh=128)
    for kw in (dict(col_h=-32), dict(col_h=128), dict(col_h=160), dict(col_h=16), dict(col_h=33),
               dict(col_h=32, ldyh=95)):
        assert _lin(h, **dict(yh, **kw)) == TB_ERR_BAD_SHAPE, kw                   # col_h in [0, N), multiple of 32
    assert _lin(h, Y=None) == TB_ERR_NULL                                            # fp32 columns need Y
    assert _lin(h, ldy=127) == TB_ERR_BAD_SHAPE                                      # ldy < n32 = N
    assert _lin(h, ldy=63, col_h=64, **yh) == TB_ERR_BAD_SHAPE                        # ldy < n32 = col_h
    assert _lin(h, Y=None, ldy=0, col_h=32, **yh) == TB_ERR_NULL
    assert _lin(h, Yh=8 * A + 1, ldyh=128) == TB_ERR_MISALIGNED                       # odd fp16 address
    assert _lin(h, prec=0, **yh) == TB_ERR_UNSUPPORTED                               # fp16 output at precision 0
    for p in (-1, 3, 4):
        assert _lin(h, prec=p) == TB_ERR_UNSUPPORTED, p                              # 3xTF32 is ops-level only
    for kw in (dict(K=132, ldx=132), dict(K=128, ldx=132), dict(X=A + 8)):            # fp16 operands: TMA needs 8 | K, ldx
        assert _lin(h, prec=2, **kw) == TB_ERR_UNSUPPORTED, kw
    for kw in (dict(K=130, ldx=132), dict(ldx=130), dict(X=A + 4), dict(W=2 * A + 4)):  # Yh has no FFMA fallback
        assert _lin(h, prec=1, **dict(yh, **kw)) == TB_ERR_UNSUPPORTED, kw


def test_linear_ln_refusals_without_gpu(handle):
    h = handle
    for k in ("X", "W", "Y", "g", "b", "out"):
        assert _ln(h, **{k: None}) == TB_ERR_NULL, k
    for kw in (dict(M=0), dict(N=0), dict(K=0), dict(ldx=127), dict(ldy=127), dict(ld_ln=127),
               dict(res=8 * A, ldr=127)):
        assert _ln(h, **kw) == TB_ERR_BAD_SHAPE, kw
    for p in (0, 3, -1):
        assert _ln(h, prec=p) == TB_ERR_UNSUPPORTED, p
    for kw in (dict(N=256, ldy=256, ld_ln=256), dict(N=64), dict(K=124, ldx=124), dict(prec=1, K=130, ldx=130),
               dict(X=A + 8)):
        assert _ln(h, **kw) == TB_ERR_UNSUPPORTED, kw                                # one n tile, TMA-able operands
    for kw in (dict(g=5 * A + 4), dict(b=6 * A + 8), dict(out=7 * A + 4), dict(out=7 * A + 2), dict(ld_ln=130),
               dict(res=8 * A + 4, ldr=128), dict(res=8 * A, ldr=130), dict(Y=4 * A + 4), dict(ldy=130),
               dict(bias=3 * A + 4)):
        assert _ln(h, **kw) == TB_ERR_MISALIGNED, kw
