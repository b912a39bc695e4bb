"""Float64 references and derived error bounds for the tensor-core projection kernel (linear_tc.cu: tb_linear
precision 1 / 2, tb_linear_ln), on CPU or device tensors. Every bound states the arithmetic it models; none is fitted
to GPU output.

Arithmetic model of linear_tc_kernel:
* Operands. kind::tf32 reads fp32 operands and multiplies their tf32 truncations (sign, exponent, 10 mantissa bits:
  `bits & -8192`, as ops._w3 splits weights for 3xTF32). kind::f16 multiplies the fp16 values as they are. A product
  of two tf32 values (11-bit significands) or two fp16 values has at most 22 significant bits: it is exact in fp32.
* Accumulation. One tcgen05.mma adds the k = 8 (tf32) / 16 (fp16) exact products of its K slice to the fp32
  accumulator, truncating (round toward zero) once per instruction (DESIGN, "Projections on tcgen05"). Modelled error
  per instruction: at most 2^-22 (two fp32 units of truncation: the aligned addends and the normalised result) of
  |accumulator| + sum |products of the slice|. Since |accumulator| <= sum |products so far| (1 + o(1)), after
  ceil(K / k) instructions |acc - exact| <= (ceil(K / k) + 2) 2^-22 sum_k |x~ w~| (the +2 absorbs the o(1) growth).
  The fused MLP chain's interpreter (tests/_chain_ref.py) uses the same model for kind::f16.
* Epilogue. fp32, in this order: + bias (grouped: the bias row of row // group), max(., 0), row mask -> 0,
  + residual, row mask -> 0. No multiply, so no FMA contraction: the result is bit-exact given the accumulator.
* fp16 outputs. cvt.rn.satfinite: clamp to +-65504, round to nearest even.
"""
import math

import numpy as np
import torch

F16_MAX = 65504.0
U32 = 2.0 ** -24  # unit roundoff of fp32 (round to nearest)


def trunc_tf32(x):
    """tf32 truncation of fp32 values: keep sign, exponent and the top 10 mantissa bits."""
    x = x.detach().float().contiguous()
    return (x.view(torch.int32) & -8192).view(torch.float32)


def sat_f16(x):
    """cvt.rn.satfinite.f16.f32 of fp32 values: clamp to +-65504, then round to nearest even."""
    return x.detach().float().clamp(-F16_MAX, F16_MAX).half()


def operands(x, w, precision):
    """The float64 values the tensor core multiplies: tf32 truncations (precision 1) or the fp16 values (precision 2)."""
    if precision == 1:
        return trunc_tf32(x).double(), trunc_tf32(w).double()
    assert precision == 2 and x.dtype == torch.float16 and w.dtype == torch.float16, (precision, x.dtype, w.dtype)
    return x.detach().double(), w.detach().double()


def acc_ref(x, w, precision):
    """float64 sum_k x~[m, k] w~[n, k] over the operands the tensor core multiplies ([M, N])."""
    xo, wo = operands(x, w, precision)
    return xo @ wo.T


def gamma_acc(K, precision):
    """(ceil(K / k) + 2) 2^-22 with k = 8 (tf32) / 16 (fp16): the accumulation model of the module docstring."""
    k = 8 if precision == 1 else 16
    return (math.ceil(K / k) + 2) * 2.0 ** -22


def acc_bound(x, w, precision):
    """Bound on |accumulator - acc_ref| per element: gamma_acc(K) sum_k |x~| |w~| ([M, N], float64)."""
    xo, wo = operands(x, w, precision)
    return gamma_acc(x.shape[1], precision) * (xo.abs() @ wo.abs().T)


def epilogue_f32(acc, bias=None, bias_group=0, relu=False, mask_pre=None, res=None, mask_post=None):
    """The kernel's epilogue on an fp32 accumulator [M, N], step by step in fp32 (IEEE round to nearest)."""
    v = acc.detach().float().clone()
    M = v.shape[0]
    if bias is not None:
        b = bias.detach().float()
        if bias_group:
            b = b.reshape(-1, v.shape[1]).repeat_interleave(bias_group, 0)[:M]
        v = v + b
    if relu:
        v = v.clamp_min(0.0)
    if mask_pre is not None:
        v[mask_pre.detach().bool()] = 0.0
    if res is not None:
        v = v + res.detach().float()
    if mask_post is not None:
        v[mask_post.detach().bool()] = 0.0
    return v


def same_bits(a, b):
    """Bit-identical fp32 / fp16 tensors on one device, +0 and -0 counted equal (NaN never equal)."""
    return a.shape == b.shape and a.dtype == b.dtype and bool((a == b).all())


def half_ulp16(a):
    """Half an fp16 ulp at magnitude a (float64 tensor; subnormal spacing 2^-24 below 2^-14)."""
    e = torch.floor(torch.log2(a.clamp_min(2.0 ** -14)))
    return 2.0 ** (e - 11)


def layernorm_ref_f64(y, gamma, beta, eps=1e-5):
    """LayerNorm over the last dim in float64 of the kernel's own fp32 rows y: (out, mean, var)."""
    y = y.detach().double()
    g, b = gamma.detach().double(), beta.detach().double()
    mu = y.mean(1, keepdim=True)
    var = ((y - mu) ** 2).mean(1, keepdim=True)
    return (y - mu) / (var + eps).sqrt() * g + b, mu, var


def ln_out_bound(y, gamma, beta, group_depth=6, eps=1e-5):
    """Bound on |ln_out - layernorm_ref_f64(y)| for the fused LayerNorm of tb_linear_ln and of the MLP chain (F_LN),
    per element of [M, 128]. Both sum each 32-column group of a row shifted by c, one of those 32 values, together
    with the squared shifted values, form S_h = 32 c + sum (y - c) and M2_h = sum (y - c)^2 - (sum (y - c))^2 / 32,
    and merge the four (S_h, M2_h) with Chan's formula. d = group_depth is the depth of the group sum sum (y - c)
    with its subtraction: 6 in tb_linear_ln (4 values per lane, then a depth-3 butterfly), 33 in the chain (one
    thread sums its 32 values in sequence); the sum of squares has depth <= d + 2. With g_k = k 2^-24 / (1 - k 2^-24),
    sigma^2 = var:
    * means: sum (y - c) is off by <= g_d sum |y - c| <= g_d 38 sqrt(M2_h), and sqrt(M2_h) <= sqrt(128) sigma; S_h adds
      one rounding of |S_h|, the row sum of the four S_h at most 3 more. So every 32-column mean and the row mean are
      off by at most e_m = g_4 max_h mean_{j in h} |y_j| + g_d 14 sigma.
    * variance: c is one of the 32 values, so (mean_h - c)^2 <= M2_h and sum (y - c)^2 <= 33 M2_h; rounding it (depth
      d + 2) and (sum (y - c))^2 / 32 (<= 2 g_d sum (y - c)^2 + one rounding of each operation) moves M2_h by
      <= g_(33 (3 d + 4)) M2_h, the merge adds g_6. A mean off by e_m moves each merge term 32 (mean_h - mean)^2 by
      64 |mean_h - mean| e_m + 64 e_m^2, and sum_h 32 |mean_h - mean| <= 128 sigma (Cauchy-Schwarz), so var moves by
      <= 8 sigma e_m + 8 e_m^2 in all.
    * rstd = 1 / sqrtf(var + eps): two more correctly rounded operations.
    * ((y - mean) rstd) gamma + beta in fp32: four roundings of at most 2^-24 of |(y - mu) r g| or |out| each.
    * fp16: a value off by e rounds to within e + half an fp16 ulp of |out| + e.
    The one-pass E[y^2] - E[y]^2 of the parent kernels exceeds this once mean / std is about 100."""
    out, mu, var = layernorm_ref_f64(y, gamma, beta, eps)
    y, g = y.detach().double(), gamma.detach().double()

    def gd(d):
        return d * U32 / (1 - d * U32)

    M, N = y.shape
    sig = var.sqrt()
    d = group_depth
    e_m = gd(4) * y.abs().reshape(M, N // 32, 32).mean(2).amax(1, keepdim=True) + gd(d) * 14 * sig
    d_var = gd(33 * (3 * d + 4) + 6) * var + 8 * sig * e_m + 8 * e_m ** 2
    s = (var + eps).sqrt()
    z = (y - mu) / s
    rel_r = d_var / (2 * (var + eps) - 2 * d_var).clamp_min(1e-300) + gd(2)
    e = g.abs() * (e_m / s + z.abs() * rel_r * (1 + e_m / s)) + 4 * U32 * ((z * g).abs() + out.abs())
    e = e * (1 + 1e-6)  # second-order products of the terms above
    return e + half_ulp16(out.abs() + e)


def _fma32(a, b, c):
    return (a.astype(np.float64) * b + c).astype(np.float32)


def _rowgroup_sum(q):
    """The store phase's 8-lane butterfly (xor 4, 2, 1) on q [M, 4 warps, 8 lanes] -> [M, 4]."""
    for k in (4, 2, 1):
        q = q.reshape(*q.shape[:2], -1, 2 * k)
        q = q[..., :k] + q[..., k:]
    return q.reshape(q.shape[0], 4)


def fused_ln_f32(y, gamma, beta, one_pass=False, eps=1e-5):
    """numpy fp32 emulation of the fused LayerNorm of tb_linear_ln in the kernel's reduction order (fp16 rows [M, 128]).
    one_pass=True: the parent kernel's var = E[y^2] - E[y]^2 from per-warp (sum, sum of squares); otherwise the
    shifted (sum, M2) partials merged with Chan's formula. Lets the CPU suite check that ln_out_bound holds for the second
    and rejects the first at large mean / std."""
    f = np.float32
    y = y.detach().cpu().float().numpy()
    M = y.shape[0]
    c = y.reshape(M, 4, 8, 4)  # [row, warp, lane (16-byte chunk), 4 columns]
    if one_pass:
        s1 = _rowgroup_sum((c[..., 0] + c[..., 1]) + (c[..., 2] + c[..., 3]))
        sq = _fma32(c[..., 0], c[..., 0], _fma32(c[..., 1], c[..., 1], _fma32(c[..., 2], c[..., 2], c[..., 3] * c[..., 3])))
        s2 = _rowgroup_sum(sq)
    else:  # shifted by the warp's first column
        d = c - c[:, :, :1, :1]
        w1 = _rowgroup_sum((d[..., 0] + d[..., 1]) + (d[..., 2] + d[..., 3]))
        w2 = _rowgroup_sum(_fma32(d[..., 0], d[..., 0], _fma32(d[..., 1], d[..., 1], _fma32(d[..., 2], d[..., 2],
                                                                                              d[..., 3] * d[..., 3]))))
        s1 = _fma32(np.full_like(w1, 32), c[:, :, 0, 0], w1)
        s2 = _fma32(-w1, w1 * f(1 / 32), w2)
    S1 = np.zeros(M, f)
    for h in range(4):
        S1 = S1 + s1[:, h]
    mean = S1 * f(1 / 128)
    if one_pass:
        S2 = np.zeros(M, f)
        for h in range(4):
            S2 = S2 + s2[:, h]
        var = np.maximum(S2 * f(1 / 128) - mean * mean, f(0))
    else:
        m2 = np.zeros(M, f)
        for h in range(4):
            dm = _fma32(s1[:, h], np.full(M, 1 / 32, f), -mean)
            m2 = _fma32(f(32) * dm, dm, m2 + s2[:, h])
        var = m2 * f(1 / 128)
    rstd = f(1) / np.sqrt(var + f(eps))
    g, b = gamma.detach().cpu().float().numpy(), beta.detach().cpu().float().numpy()
    out = ((y - mean[:, None]) * rstd[:, None]) * g + b
    return torch.from_numpy(out.astype(np.float32)).half()
