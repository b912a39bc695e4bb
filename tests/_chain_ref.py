"""Float64 reference of a fused MLP chain program (tb_chain_encode / tb_chain_run, include/tb_knarpe.h), the encoder's
rules re-derived in Python, and a seeded generator of random programs the encoder must accept.

A program is a `ChainProgram.spec`: a list of plain dicts, {"kind": "load", src, lds, out_buf, src_col, f16} or
{"kind": "gemm", w [N, K], a_bufs, bias, n0, relu, out_buf, mask_pre, mask_post, res, ldr, res_col, out_g, ldg, g_col,
n_valid, out_h, ldh, h_col, ln_out, ld_ln, ln_gamma, ln_beta} (indices -1 = unused, n_valid 0 = 128). Bindings are
row-major tensors [rows, ld] (masks: [rows])."""
import math
import random

import torch

F16_MAX = 65504.0
MAX_UNITS, MAX_MAPS, MAX_BIND = 32, 24, 16
SMEM_MAX, BUF_BYTES, WSTAGE_BYTES, UNIT_BYTES = 227 * 1024, 2 * 128 * 128, 128 * 128, 192
TB_OK, TB_ERR_BAD_SHAPE, TB_ERR_UNSUPPORTED, TB_ERR_MISALIGNED, TB_ERR_NULL = 0, -1, -3, -4, -5


def f16(x):
    """cvt.rn.satfinite.f16.f32: clamp to the largest finite half, then round to nearest even."""
    return x.clamp(-F16_MAX, F16_MAX).float().half().to(x.dtype)


def ulp16(x):
    """Spacing of fp16 numbers at |x| (2^-24 below the normal range)."""
    _, e = torch.frexp(x.abs().clamp_min(2.0 ** -14))
    return torch.ldexp(torch.ones_like(x), (e - 11).clamp_min(-24))


# ---------------------------------------------------------------------------------------------------- encoder rules
def tail_bytes(n_units):
    """Shared memory of the unit table, biases, LayerNorm partials, bindings, mbarriers and TMEM slot (mlp_chain.cu)."""
    return n_units * UNIT_BYTES + n_units * 512 + 4 * 128 * 8 + MAX_BIND * 8 + (16 + 2 * MAX_UNITS) * 8 + 64


def ring_depth(n_buf, n_units):
    """Weight stages the encoder gives a program: what shared memory leaves after the buffers, at most 8."""
    return min(8, (SMEM_MAX - 1024 - n_buf * BUF_BYTES - tail_bytes(n_units)) // WSTAGE_BYTES)


def _aligned16(t):
    return t is None or t.data_ptr() % 16 == 0


def encode_rules(spec, n_buf):
    """What tb_chain_encode returns for `spec`, in the order it checks: dict(code, n_stage, n_maps, waits) where
    waits[u] lists the units GEMM u waits for (last writer of each input buffer, then the GEMM 4 earlier)."""
    out = dict(code=TB_OK, n_stage=0, n_maps=0, waits=[[] for _ in spec])
    n = len(spec)
    if n <= 0 or n > MAX_UNITS or n_buf < 2 or n_buf > 5:
        return dict(out, code=TB_ERR_BAD_SHAPE)
    out["n_stage"] = ring_depth(n_buf, n)
    if out["n_stage"] < 2:
        return dict(out, code=TB_ERR_UNSUPPORTED)
    maps, writer, gemms = [], [-1] * 8, []
    bad_bind = lambda b: b < -1 or b >= MAX_BIND - 1  # noqa: E731
    for u, s in enumerate(spec):
        if s["out_buf"] >= n_buf:
            return dict(out, code=TB_ERR_BAD_SHAPE)
        binds = ("src",) if s["kind"] == "load" else ("mask_pre", "mask_post", "res", "out_g", "out_h", "ln_out")
        if any(bad_bind(s[k]) for k in binds):
            return dict(out, code=TB_ERR_BAD_SHAPE)
        if s["kind"] == "load":
            if s["src"] < 0 or s["out_buf"] < 0 or (s["lds"] | s["src_col"]) & (7 if s["f16"] else 3):
                return dict(out, code=TB_ERR_BAD_SHAPE)
        else:
            N, K = s["w"].shape
            if K % 64 or K // 64 > 8 or s["n0"] < 0 or s["n0"] >= N or s["n_valid"] > 128:
                return dict(out, code=TB_ERR_BAD_SHAPE)
            if (not _aligned16(s["w"]) or not _aligned16(s["bias"]) or (s["res"] >= 0 and (s["ldr"] | s["res_col"]) & 3)
                    or (s["out_h"] >= 0 and (s["ldh"] | s["h_col"]) & 7)
                    or (s["ln_out"] >= 0 and (s["ld_ln"] & 7 or s["ln_gamma"] is None or s["ln_beta"] is None
                                              or not _aligned16(s["ln_gamma"]) or not _aligned16(s["ln_beta"])))):
                return dict(out, code=TB_ERR_MISALIGNED)
            key = (s["w"].data_ptr(), K, N)
            if key not in maps:
                if len(maps) == MAX_MAPS:
                    return dict(out, code=TB_ERR_UNSUPPORTED)
                maps.append(key)
            waits = out["waits"][u]
            for kb in range(K // 64):
                b = s["a_bufs"][kb // 2]
                if b < 0 or b >= n_buf or writer[b] < 0:
                    return dict(out, code=TB_ERR_BAD_SHAPE)
                if writer[b] not in waits:
                    waits.append(writer[b])
            if len(gemms) >= 4 and gemms[-4] not in waits:
                waits.append(gemms[-4])
            if len(waits) > 6:
                return dict(out, code=TB_ERR_UNSUPPORTED)
            gemms.append(u)
        if s["out_buf"] >= 0:
            writer[s["out_buf"]] = u
    out["n_maps"] = len(maps)
    return out


# ---------------------------------------------------------------------------------------------------- interpreter
def _cols(x, c0, n):
    return x[:, c0:c0 + n]


def interpret(spec, bind, rows, round16=True, bound=False):
    """Runs `spec` in program order on rows `rows` (a LongTensor of row indices < M) of the bindings, in float64.
    Returns (X, E, V): X[i] the float64 rows of binding i after the program (masks: bool), E[i] an upper bound of
    |kernel - X| on everything the program wrote (0 elsewhere; with bound=True), V[u] = (v, bound) of GEMM u's epilogue
    value. round16: every buffer write, fp32 LOAD, out_h and ln_out is rounded like cvt.rn.satfinite.f16.
    The bound carries, unit by unit: the MMA's fp32 accumulation ((K/16 + 2) 2^-22 sum|a w|), the fp32 bias / residual
    adds (2^-23 of the operands), fp16 rounding (a value off by e may round to a half one ulp away: e + ulp16) and the
    input error through |W|; a LayerNorm row through its mean and standard deviation."""
    X, E = {}, {}
    for i, t in enumerate(bind):
        if t is None:
            continue
        t = t.detach().cpu()
        if t.dtype in (torch.bool, torch.uint8):
            X[i] = t.reshape(-1)[rows] != 0
        else:
            X[i] = t.reshape(t.shape[0], -1)[rows].double()
            E[i] = torch.zeros_like(X[i])
    R = len(rows)
    rnd = f16 if round16 else (lambda x: x)  # noqa: E731
    bufs, ebufs, V = {}, {}, {}
    for u, s in enumerate(spec):
        if s["kind"] == "load":
            bufs[s["out_buf"]] = rnd(_cols(X[s["src"]], s["src_col"], 128))
            ebufs[s["out_buf"]] = torch.zeros(R, 128, dtype=torch.float64)
            continue
        W = s["w"].detach().cpu().double()
        N, K = W.shape
        n0 = s["n0"]
        Wt = torch.zeros(128, K, dtype=torch.float64)
        Wt[:min(128, N - n0)] = W[n0:n0 + 128]
        A = torch.cat([_cols(bufs[s["a_bufs"][kb // 2]], 64 * (kb % 2), 64) for kb in range(K // 64)], 1)
        EA = torch.cat([_cols(ebufs[s["a_bufs"][kb // 2]], 64 * (kb % 2), 64) for kb in range(K // 64)], 1)
        b = torch.zeros(128, dtype=torch.float64)
        if s["bias"] is not None:
            bb = s["bias"].detach().cpu().double().reshape(-1)[n0:n0 + 128]
            b[:bb.numel()] = bb
        acc = A @ Wt.T
        v = acc + b
        P = EA @ Wt.abs().T
        ev = P + (K / 16 + 2) * 2.0 ** -22 * (A.abs() @ Wt.abs().T + P) + 2.0 ** -23 * (acc.abs() + P + b.abs())
        if s["relu"]:
            v = v.clamp_min(0.0)
        if s["mask_pre"] >= 0:
            m = X[s["mask_pre"]]
            v[m], ev[m] = 0.0, 0.0
        if s["res"] >= 0:
            v = v + _cols(X[s["res"]], s["res_col"], 128)
            ev = ev + _cols(E[s["res"]], s["res_col"], 128) + 2.0 ** -23 * (v.abs() + ev)
        if s["mask_post"] >= 0:
            m = X[s["mask_post"]]
            v[m], ev[m] = 0.0, 0.0
        V[u] = (v, ev)
        nv = s["n_valid"] or 128
        eh = ev + ulp16(v.abs() + ev) if round16 else ev
        if s["out_buf"] >= 0:
            bufs[s["out_buf"]], ebufs[s["out_buf"]] = rnd(v), eh
        if s["out_g"] >= 0:
            _cols(X[s["out_g"]], s["g_col"], nv)[:] = v[:, :nv]
            _cols(E[s["out_g"]], s["g_col"], nv)[:] = ev[:, :nv]
        if s["out_h"] >= 0:
            _cols(X[s["out_h"]], s["h_col"], nv)[:] = rnd(v[:, :nv])
            _cols(E[s["out_h"]], s["h_col"], nv)[:] = eh[:, :nv]
        if s["ln_out"] >= 0:
            g = s["ln_gamma"].detach().cpu().double().reshape(-1)[:128]
            be = s["ln_beta"].detach().cpu().double().reshape(-1)[:128]
            mu = v.mean(1, keepdim=True)
            var = ((v - mu) ** 2).mean(1, keepdim=True)
            sig = (var + 1e-5).sqrt()
            z = (v - mu) / sig
            y = z * g + be
            # input error: mean and every column move by <= e_r, the variance by <= 2 sigma e_r + e_r^2. The kernel's
            # fp32 statistics (per 32 columns: sequential sums of v - c and (v - c)^2, c the first of them, then Chan's
            # merge; tests/_linear_ref.ln_out_bound derives the same terms for depth-8 sums): every mean off by
            # <= e_s = 2^-24 (130 max|v| + 470 sigma), the variance by 2^-24 3400 var + 8 sigma e_s + 8 e_s^2
            e_r = ev.amax(1, keepdim=True)
            sd = var.sqrt() + e_r
            e_s = 2.0 ** -24 * (130 * (v.abs().amax(1, keepdim=True) + e_r) + 470 * sd)
            d_var = 2 * var.sqrt() * e_r + e_r ** 2 + 2.0 ** -24 * 3400 * sd ** 2 + 8 * sd * e_s + 8 * e_s ** 2
            d_mu = e_r + 2.0 ** -24 * 130 * (v.abs().mean(1, keepdim=True) + e_r)
            ey = g.abs() * ((ev + d_mu) / sig + z.abs() * d_var / (var + 1e-5)) + 2.0 ** -21 * (y.abs() + (z * g).abs())
            ey = 2 * ey + ulp16(y.abs() + 2 * ey) if round16 else 2 * ey
            X[s["ln_out"]][:, :128] = rnd(y)
            E[s["ln_out"]][:, :128] = ey
    return X, E, V


def written_mask(spec, bind_idx, shape, M):
    """bool [rows, ld] of the elements of binding `bind_idx` the program writes for M rows."""
    w = torch.zeros(shape, dtype=torch.bool)
    for s in spec:
        if s["kind"] != "gemm":
            continue
        nv = s["n_valid"] or 128
        if s["out_g"] == bind_idx:
            w[:M, s["g_col"]:s["g_col"] + nv] = True
        if s["out_h"] == bind_idx:
            w[:M, s["h_col"]:s["h_col"] + nv] = True
        if s["ln_out"] == bind_idx:
            w[:M, :128] = True
    return w


# ---------------------------------------------------------------------------------------------------- generator
# Binding layout of the generated programs (the split run of a program adds up to 5 buffer tensors and a probe after
# these, so the original programs use indices 0..8 only):
#   0 X32 fp32 [M, 264] LOAD source; 1 X16 fp16 [M, 272] LOAD source; 2, 3 row masks u8 [M]; 4 RES fp32 [M, 260];
#   5 GV fp32 [M, 400]: out_g slots at columns 4, 136, 268 (vector path), also read back as residual rows;
#   6 GS fp32 [M, 267]: out_g slots at columns 1, 133 (odd pitch and column: scalar path);
#   7 H fp16 [M, 280]: out_h slots at columns 8, 144; 8 LN fp16 [M, 136]: ln_out.
LAYOUT = [("X32", torch.float32, 264), ("X16", torch.float16, 272), ("MA", torch.uint8, 0), ("MB", torch.uint8, 0),
          ("RES", torch.float32, 260), ("GV", torch.float32, 400), ("GS", torch.float32, 267),
          ("H", torch.float16, 280), ("LN", torch.float16, 136)]
SLOTS = {5: [4, 136, 268], 6: [1, 133], 7: [8, 144]}
N_VALID = (1, 6, 31, 32, 33, 127, 128)
SENTINEL32, SENTINEL16 = 0x7FBADBAD, 0x7E5A  # NaN bit patterns in never-written output columns


def make_bindings(M, seed):
    """CPU tensors of LAYOUT for M rows: inputs and GV random (GV is also a residual source), other outputs sentinel."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for i, (name, dt, ld) in enumerate(LAYOUT):
        if dt == torch.uint8:
            out.append((torch.rand(M, generator=g) < 0.3).to(torch.uint8))
        elif name in ("X32", "X16", "RES", "GV"):
            out.append(torch.randn(M, ld, generator=g).to(dt))
        elif dt == torch.float32:
            out.append(torch.full((M, ld), SENTINEL32, dtype=torch.int32).view(torch.float32))
        else:
            out.append(torch.full((M, ld), SENTINEL16, dtype=torch.int16).view(torch.float16))
    return out


def _unit(kind, **kw):
    base = dict(out_buf=-1) if kind == "load" else dict(
        bias=None, n0=0, relu=False, out_buf=-1, mask_pre=-1, mask_post=-1, res=-1, ldr=0, res_col=0, out_g=-1, ldg=0,
        g_col=0, n_valid=0, out_h=-1, ldh=0, h_col=0, ln_out=-1, ld_ln=0, ln_gamma=None, ln_beta=None)
    base.update(kind=kind, **kw)
    return base


def load_unit(rng, buf):
    if rng.random() < 0.5:
        return _unit("load", src=1, lds=272, out_buf=buf, src_col=8 * rng.randint(0, 18), f16=True)
    return _unit("load", src=0, lds=264, out_buf=buf, src_col=4 * rng.randint(0, 34), f16=False)


def gen_program(seed, n_buf=None, n_units=None, long_run=False):
    """A random program the encoder must accept: (spec, n_buf). Weights are CPU fp16 tensors [N, K] shared between
    units (same tensor, same K) to exercise the map de-duplication; at most 24 distinct ones."""
    rng = random.Random(seed)
    gw = torch.Generator().manual_seed(seed)
    n_buf = n_buf or rng.randint(2, 5)
    n_units = n_units or rng.randint(1, 32)
    p_load = 0.0 if long_run else 0.15
    spec, pool, written = [], [], set()
    free = {k: list(v) for k, v in SLOTS.items()}
    gv_used, ln_used = [], False
    for u in range(n_units):
        if not written or (rng.random() < p_load and u < n_units - 1):
            b = rng.randrange(n_buf)
            spec.append(load_unit(rng, b))
            written.add(b)
            continue
        K = 64 * rng.randint(1, 8)
        same_k = [w for w in pool if w.shape[1] == K]
        if len(pool) == MAX_MAPS and not same_k:
            w = rng.choice(pool)
            K = w.shape[1]
        elif same_k and (rng.random() < 0.35 or len(pool) == MAX_MAPS):
            w = rng.choice(same_k)
        else:
            N = rng.choice([6, 64, 100, 128, 200, 256, 384])
            w = (torch.randn(N, K, generator=gw) / math.sqrt(K)).half()
            pool.append(w)
        N = w.shape[0]
        a_bufs = [rng.choice(sorted(written)) for _ in range((K + 127) // 128)]
        s = _unit("gemm", w=w, a_bufs=a_bufs, n0=rng.choice([n for n in (0, 64, 128, 200, 256) if n < N]),
                  relu=rng.random() < 0.6)
        if rng.random() < 0.7:
            s["bias"] = torch.randn(N, generator=gw) * 0.2
        if rng.random() < 0.2:
            s["mask_pre"] = rng.choice([2, 3])
        if rng.random() < 0.2:
            s["mask_post"] = rng.choice([2, 3])
        if rng.random() < 0.25:
            if gv_used and rng.random() < 0.6:  # an earlier unit's out_g, same columns: the allowed aliasing
                s.update(res=5, ldr=400, res_col=rng.choice(gv_used))
            else:
                s.update(res=4, ldr=260, res_col=4 * rng.randint(0, 33))
        if rng.random() < 0.85:
            s["out_buf"] = rng.randrange(n_buf)
        if rng.random() < 0.25:
            b = rng.choice([5, 6])
            if free[b]:
                col = free[b].pop(rng.randrange(len(free[b])))
                s.update(out_g=b, ldg=LAYOUT[b][2], g_col=col)
                if b == 5:
                    gv_used.append(col)
        if rng.random() < 0.2 and free[7]:
            s.update(out_h=7, ldh=280, h_col=free[7].pop(rng.randrange(len(free[7]))))
        if s["out_g"] >= 0 or s["out_h"] >= 0:
            s["n_valid"] = rng.choice(N_VALID)
        if rng.random() < 0.08 and not ln_used:
            ln_used = True
            s.update(ln_out=8, ld_ln=136, ln_gamma=torch.rand(128, generator=gw) + 0.5,
                     ln_beta=torch.randn(128, generator=gw) * 0.1)
        if s["out_buf"] < 0 and s["out_g"] < 0 and s["out_h"] < 0 and s["ln_out"] < 0:
            s["out_buf"] = rng.randrange(n_buf)
        spec.append(s)
        if s["out_buf"] >= 0:
            written.add(s["out_buf"])
    return spec, n_buf


def max_wait_program():
    """n_buf 5: a K = 512 GEMM over 4 buffers with 4 different last writers and, 4 GEMMs back, a 5th unit that wrote
    none of them: 5 waits, the most any unit can have."""
    rng = random.Random(5)
    gw = torch.Generator().manual_seed(5)
    w = lambda n, k: (torch.randn(n, k, generator=gw) / math.sqrt(k)).half()  # noqa: E731
    spec = [load_unit(rng, b) for b in range(4)]
    spec += [_unit("gemm", w=w(128, 128), a_bufs=[0], out_buf=1, relu=True),
             _unit("gemm", w=w(128, 128), a_bufs=[1], out_buf=4),
             _unit("gemm", w=w(128, 128), a_bufs=[0], out_buf=2, relu=True),
             _unit("gemm", w=w(128, 128), a_bufs=[2], out_buf=3, relu=True),
             _unit("gemm", w=w(128, 128), a_bufs=[3], out_h=7, ldh=280, h_col=8, n_valid=33),
             _unit("gemm", w=w(100, 512), a_bufs=[0, 1, 2, 3], bias=torch.randn(100, generator=gw), out_g=5, ldg=400,
                   g_col=136)]
    return spec, 5


# The random programs of tests/test_mlp_chain_gpu.py: (seed, n_buf, n_units, long_run). n_buf cycles through 2..5 and
# the unit counts straddle the 19 / 20 boundary of the ring-depth table, so every depth 2..8 runs; every fifth program
# is one LOAD followed by GEMMs only (TMEM regions reused up to 7 times per tile).
PROGRAMS = [(1000 + i, 2 + i % 4, (1, 3, 8, 19, 20, 26, 32, 13)[(i // 4) % 8], i % 5 == 4) for i in range(64)]


def fan_out_program():
    """n_buf 2: one LOAD, then 8 GEMMs that all read that buffer and write only global outputs. Their input's writer
    finished long ago, so from the 5th GEMM on the only thing keeping a unit's MMAs out of a TMEM region is its wait for
    the epilogue of the GEMM 4 earlier (the regions are used in turn): without it the later units overwrite
    accumulators the earlier ones' epilogues are still reading."""
    rng = random.Random(9)
    gw = torch.Generator().manual_seed(9)
    outs = [dict(out_g=5, ldg=400, g_col=c) for c in SLOTS[5]] + [dict(out_g=6, ldg=267, g_col=c) for c in SLOTS[6]]
    outs += [dict(out_h=7, ldh=280, h_col=c) for c in SLOTS[7]]
    outs += [dict(ln_out=8, ld_ln=136, ln_gamma=torch.rand(128, generator=gw) + 0.5, ln_beta=torch.randn(128, generator=gw))]
    spec = [load_unit(rng, 0)]
    for o in outs:
        spec.append(_unit("gemm", w=(torch.randn(128, 128, generator=gw) / 11.3).half(), a_bufs=[0],
                          bias=torch.randn(128, generator=gw) * 0.2, relu=True, **o))
    return spec, 2
