"""GPU: the fused MLP chain (tb_chain_encode / tb_chain_run) program by program.

* Random programs (tests/_chain_ref.py: n_buf 2..5, 1..32 units, every ring depth 2..8, K = 64..512, every epilogue
  flag) run fused and as a chain of one-GEMM sub-programs whose buffers pass through fp16 global tensors. The MMA
  sequence, the fp16 bits and the epilogue code are the same, so every output must be bit-identical: any dependency,
  weight-ring or TMEM-reuse race shows up here without a tolerance.
* Each GEMM's fp32 epilogue value (from the split run, on the kernel's own fp16 inputs) against float64, within
  (K/16 + 2) 2^-22 sum|a w| + 2^-23 (|acc| + |bias| + |v|): a dropped k-block, a wrong n0 slice, swizzle chunk or bias
  offset misses by orders of magnitude.
* The whole fused program against the float64 interpreter, within a bound propagated unit by unit (each fp16 rounding
  may land one ulp away and that difference travels through |W| to every later unit).
* Guard columns and rows, LOAD sources untouched, M sweeps across tile and wave boundaries, the engine's head chain and
  FFN program, every encoder refusal, the run-time binding checks and the fp16 range guard.
No test here launches an invalid program: every refusal is returned before the launch (tests/test_mlp_chain_cpu.py
checks the run-time refusals on a hand-made program without any device first)."""
import ctypes
import struct

import pytest
import torch

import _chain_ref as CR
import _linear_ref as LR
from oracle import tb_oracle as O
from trafficbotsv1_5_b200 import config, params

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from trafficbotsv1_5_b200 import lib as L
    from trafficbotsv1_5_b200 import ops
    from trafficbotsv1_5_b200.model import HotPathModel

DEV = "cuda"
GEMM_KEYS = ("bias", "n0", "relu", "out_buf", "mask_pre", "mask_post", "res", "ldr", "res_col", "out_g", "ldg", "g_col",
             "n_valid", "out_h", "ldh", "h_col", "ln_out", "ld_ln", "ln_gamma", "ln_beta")
OUTS = (5, 6, 7, 8)                 # output bindings of the generated programs
SPLIT_T, SPLIT_BIND = 9, 15         # split run: buffer tensors from binding 9, then the probe and the new buffer
M_CYCLE = (1, 100, 128, 129, 700, 1500, 2900)
STATS = dict(worst_unit=0.0, worst_prog=0.0, depths=set(), bufs=set(), flags=set(), programs=0)


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


def _same(a, b):
    """Bit-identical (NaN sentinels included)."""
    a, b = a.cpu(), b.cpu()
    return a.dtype == b.dtype and (torch.equal(a, b) if a.dtype == torch.uint8 else torch.equal(_bits(a), _bits(b)))


def _n_stage(p):
    return struct.unpack_from("<4i", bytes(p.host))[3]


def _build(spec, n_buf, wcache):
    p = ops.ChainProgram(DEV, n_buf)
    for s in spec:
        if s["kind"] == "load":
            p.load(s["src"], s["lds"], s["out_buf"], s["src_col"], s["f16"])
        else:
            w = wcache.setdefault(s["w"].data_ptr(), s["w"].to(DEV))
            p.gemm(w, s["a_bufs"], **{k: s[k] for k in GEMM_KEYS})
    return p.finish()


def _split(spec, n_buf, binds, M, wcache):
    """Runs `spec` one GEMM at a time on the device tensors `binds` (updated in place). A LOAD becomes an fp16 tensor
    (cvt.rn.satfinite = clamp + round to nearest even); a GEMM is a sub-program LOADing its fp16 input tensors into the
    same buffers, run up to three times: fp32 epilogue value -> probe, buffer output -> a fresh fp16 tensor (out_h of all
    128 columns), then the unit's own global outputs. Returns {u: (probe, per-unit reference bindings)}."""
    T, units = {}, {}
    for u, s in enumerate(spec):
        if s["kind"] == "load":
            src = binds[s["src"]][:, s["src_col"]:s["src_col"] + 128]
            T[s["out_buf"]] = (src if s["f16"] else src.clamp(-CR.F16_MAX, CR.F16_MAX).half()).contiguous().clone()
            continue
        used = sorted(set(s["a_bufs"]))
        probe = torch.empty(M, 128, device=DEV)
        newbuf = torch.empty(M, 128, dtype=torch.float16, device=DEV)
        extra = [None] * (SPLIT_T - len(binds)) + [T[b] for b in used] + [None] * (4 - len(used)) + [probe, newbuf]
        b_all = binds + extra
        assert len(b_all) == SPLIT_BIND
        # inputs of the per-unit reference, as the unit sees them (masks, residual rows before its own writes)
        ref_b = [None] * SPLIT_BIND
        for i in (s["mask_pre"], s["mask_post"], s["res"]):
            if i >= 0:
                ref_b[i] = b_all[i].cpu()
        for j, b in enumerate(used):
            ref_b[SPLIT_T + j] = T[b].cpu()
        ref_b[13] = torch.zeros(M, 128)
        ref_spec = [CR._unit("load", src=SPLIT_T + j, lds=128, out_buf=b, src_col=0, f16=True) for j, b in enumerate(used)]
        base = {k: s[k] for k in GEMM_KEYS}
        base.update(out_buf=-1, out_g=-1, out_h=-1, ln_out=-1)
        ref_spec.append(dict(base, kind="gemm", w=s["w"], a_bufs=s["a_bufs"], out_g=13, ldg=128, g_col=0, n_valid=128))

        def sub(**over):
            p = ops.ChainProgram(DEV, n_buf)
            for j, b in enumerate(used):
                p.load(SPLIT_T + j, 128, b, f16=True)
            p.gemm(wcache.setdefault(s["w"].data_ptr(), s["w"].to(DEV)), s["a_bufs"], **dict(base, **over))
            p.finish().run(b_all, M)

        sub(out_g=13, ldg=128, g_col=0, n_valid=128)
        if s["out_buf"] >= 0:
            sub(out_h=14, ldh=128, h_col=0, n_valid=128)
        if s["out_g"] >= 0 or s["out_h"] >= 0 or s["ln_out"] >= 0:
            sub(**{k: s[k] for k in ("out_g", "ldg", "g_col", "n_valid", "out_h", "ldh", "h_col", "ln_out", "ld_ln")})
        if s["out_buf"] >= 0:
            T[s["out_buf"]] = newbuf
        units[u] = (probe, ref_spec, ref_b)
    return units


def _check_vs_interpreter(spec, init, out, M, rows, what):
    """Fused outputs `out` (device) against the interpreter on the inputs `init` (CPU): inside what the program writes
    within the propagated bound, everything else bit-identical to `init`. Returns the worst error / bound."""
    X, E, _ = CR.interpret(spec, init, rows, bound=True)
    worst = 0.0
    for i in OUTS:
        got = out[i].cpu()
        wm = CR.written_mask(spec, i, got.shape, M)
        assert torch.equal(_bits(got)[~wm], _bits(init[i])[~wm]), f"{what}: binding {i} written outside its columns / rows"
        g, e, x, w = got[rows].double(), E[i], X[i], wm[rows]
        if bool(w.any()):
            err = (g - x).abs()[w]
            lim = e[w] + 1e-300
            assert bool(torch.isfinite(g[w]).all()), f"{what}: binding {i} has non-finite values"
            assert bool((err <= lim).all()), (f"{what}: binding {i}: {int((err > lim).sum())} values out of bound, worst "
                                              f"{float((err / lim).max()):.3g} x bound")
            worst = max(worst, float((err / lim).max()))
    for i in range(5):  # LOAD sources, masks, residual rows
        assert _same(out[i], init[i]), f"{what}: input {i} changed"
    return worst


def _flags(spec):
    f = set()
    for s in spec:
        if s["kind"] == "load":
            f.add("load_f16" if s["f16"] else "load_f32")
            continue
        for k in ("mask_pre", "mask_post", "res", "out_buf", "out_h", "ln_out"):
            if s[k] >= 0:
                f.add(k)
        if s["out_g"] >= 0:
            f.add("out_g_vector" if (s["ldg"] | s["g_col"]) % 4 == 0 else "out_g_scalar")
        if s["res"] == 5:
            f.add("res_reads_out_g")
    return f


@pytest.mark.parametrize("case", range(len(CR.PROGRAMS)))
def test_random_program_fused_equals_split_and_float64(case):
    seed, n_buf, n_units, long_run = CR.PROGRAMS[case]
    spec, n_buf = CR.gen_program(seed, n_buf, n_units, long_run)
    M = M_CYCLE[case % len(M_CYCLE)]
    wc = {}
    p = _build(spec, n_buf, wc)
    assert _n_stage(p) == CR.ring_depth(n_buf, len(spec))
    init = CR.make_bindings(M, seed)
    fused = [t.to(DEV) for t in init]
    n0 = ops.LAUNCHES
    p.run(fused, M)
    assert ops.LAUNCHES == n0 + 1
    split = [t.to(DEV) for t in init]
    units = _split(spec, n_buf, split, M, wc)
    torch.cuda.synchronize()
    for i in range(len(init)):
        assert _same(fused[i], split[i]), f"program {seed}: binding {i} differs between the fused and the split run"
    # every GEMM against float64 on its own fp16 inputs
    rows = torch.arange(M)
    for u, (probe, ref_spec, ref_b) in units.items():
        X, E, _ = CR.interpret(ref_spec, ref_b, rows, bound=True)
        err, lim = (probe.cpu().double() - X[13]).abs(), E[13] + 1e-300
        r = float((err / lim).max())
        assert r <= 1.0, f"program {seed}, unit {u}: {int((err > lim).sum())} values out of bound, worst {r:.3g} x bound"
        STATS["worst_unit"] = max(STATS["worst_unit"], r)
    STATS["worst_prog"] = max(STATS["worst_prog"], _check_vs_interpreter(spec, init, fused, M, rows, f"program {seed}"))
    STATS["depths"].add(_n_stage(p))
    STATS["bufs"].add(n_buf)
    STATS["flags"] |= _flags(spec)
    STATS["programs"] += 1
    if STATS["programs"] == len(CR.PROGRAMS):
        print(f"\nchain programs: {STATS['programs']}, ring depths {sorted(STATS['depths'])}, n_buf {sorted(STATS['bufs'])}, "
              f"flags {sorted(STATS['flags'])}, worst unit error {STATS['worst_unit']:.3g} of its bound, worst "
              f"program output {STATS['worst_prog']:.3g} of its bound")


@pytest.mark.parametrize("M", [1000, 2 * 148 * 128 + 5])
def test_fan_out_reuses_tmem_regions(M):
    """Eight GEMMs on one LOADed buffer, outputs only (tests/_chain_ref.fan_out_program): only the TMEM-region wait
    orders a unit's MMAs after the epilogue of the unit 4 earlier. Fused equals split bit for bit and agrees with the
    interpreter."""
    spec, n_buf = CR.fan_out_program()
    waits = CR.encode_rules(spec, n_buf)["waits"]
    assert all(w == [0, u - 4] for u, w in enumerate(waits) if u >= 5)  # the LOAD + the GEMM 4 earlier
    wc = {}
    init = CR.make_bindings(M, 9)
    fused, split = [t.to(DEV) for t in init], [t.to(DEV) for t in init]
    _build(spec, n_buf, wc).run(fused, M)
    _split(spec, n_buf, split, M, wc)
    for i in OUTS:
        assert _same(fused[i], split[i]), i
    _check_vs_interpreter(spec, init, fused, M, torch.arange(0, M, 7), f"fan-out M = {M}")


def test_max_wait_unit():
    """The unit with the most waits a program can give (4 input-buffer writers + the GEMM 4 earlier = 5) runs fused
    exactly as split; no unit can reach a 6th wait, so the encoder's 7th-wait refusal has no program that triggers it."""
    spec, n_buf = CR.max_wait_program()
    assert max(len(w) for w in CR.encode_rules(spec, n_buf)["waits"]) == 5
    M, wc = 1000, {}
    init = CR.make_bindings(M, 5)
    fused, split = [t.to(DEV) for t in init], [t.to(DEV) for t in init]
    _build(spec, n_buf, wc).run(fused, M)
    _split(spec, n_buf, split, M, wc)
    for i in OUTS:
        assert torch.equal(_bits(fused[i]), _bits(split[i])), i
    _check_vs_interpreter(spec, init, fused, M, torch.arange(M), "max-wait program")


@pytest.mark.parametrize("M", [1, 127, 128, 129, 148 * 128, 148 * 128 + 1, 3 * 148 * 128 + 77])
def test_m_sweep_guards(M):
    """One program with every output kind (fp32 / fp16 LOADs, out_g on both paths, out_h, ln_out, a residual that reads
    an earlier out_g) across tile and wave boundaries: sentinel-filled outputs are written only at rows < M and inside
    [g_col, g_col + n_valid) / [h_col, h_col + n_valid) / [0, 128), LOAD sources and residual inputs are untouched,
    sampled rows agree with the interpreter, and a run on the first M' < M rows gives the same bits there."""
    spec, n_buf = CR.gen_program(60, 4, 20)
    f = _flags(spec)
    assert {"load_f16", "load_f32", "out_g_vector", "out_g_scalar", "out_h", "ln_out", "res_reads_out_g"} <= f, f
    p = _build(spec, n_buf, {})
    init = CR.make_bindings(M, M)
    out = [t.to(DEV) for t in init]
    p.run(out, M)
    g = torch.Generator().manual_seed(M)
    edges = [r for r in (0, 1, 126, 127, 128, 129, 148 * 128 - 1, 148 * 128, M - 2, M - 1) if 0 <= r < M]
    rows = torch.unique(torch.cat([torch.tensor(edges, dtype=torch.long), torch.randint(0, M, (256,), generator=g)]))
    _check_vs_interpreter(spec, init, out, M, rows, f"M = {M}")
    if M > 1:
        Mp = M // 2 if M > 300 else M - 1
        part = [t.to(DEV) for t in init]
        p.run(part, Mp)
        for i in OUTS:
            assert torch.equal(_bits(part[i][:Mp]), _bits(out[i][:Mp])), i
            assert torch.equal(_bits(part[i][Mp:]).cpu(), _bits(init[i][Mp:])), i


# ------------------------------------------------------------------------------------------------ the engine's programs
def _model():
    cfg = config.default_model_cfg()
    P = params.init_params(cfg, 0)
    return HotPathModel(P, cfg, config.derived_sizes(cfg), DEV, precision=1), P, cfg


def test_engine_heads_chain_vs_oracle_and_interpreter():
    """HotPathModel.heads on one seeded state of the rollout-small shape (2 scenes x 3 rollouts x 32 agents), fused
    (opt["chain"]) and per layer, against the oracle's navi_encoder.mlp_pe -> add_navi_latent x 2 -> action-head
    branches in float64. DESIGN §3 gives 2.3e-4 (chain) and 4.3e-4 (separate launches) against the fp32 path on real
    rollouts; fp16 activations round by 2^-11 relative at each of 13 layers, so both must stay within 4e-3 of the output
    scale. The interpreter, run on the program's own spec and inputs, bounds the fused result tightly."""
    m, P, cfg = _model()
    d, M = cfg["hidden_dim"], 2 * 3 * 32
    g = torch.Generator().manual_seed(17)
    x_cat = torch.cat([torch.randn(M, d, generator=g), torch.zeros(M, d)], 1).to(DEV)
    st = dict(pose=(torch.randn(M, 3, generator=g) * torch.tensor([30.0, 30.0, 2.0])).to(DEV),
              navi_invalid=(torch.rand(M, generator=g) < 0.2).to(DEV),
              latent_invalid=(torch.rand(M, generator=g) < 0.2).to(DEV),
              latent=torch.randn(M, P["add_latent.mlp_in.fc_layers.0.weight"].shape[1], generator=g).to(DEV))
    navi_pose = (torch.randn(M, 3, generator=g) * torch.tensor([60.0, 60.0, 2.0])).to(DEV)
    feat = (torch.randn(M, d, generator=g) * 0.5).to(DEV)
    zl = torch.relu(torch.randn(M, d, generator=g)).masked_fill(st["latent_invalid"].cpu()[:, None], 0.0)
    pe = ops.pose_emb(navi_pose, m.freq_rpe, d, frame=st["pose"], frame_div=1).cpu().double()
    P64 = {k: v.double() for k, v in P.items()}
    nf = feat.cpu().double() + O.mlp(P64, "navi_encoder.mlp_pe", pe, (0,), False)
    x2 = O.add_navi_latent(P64, "add_navi", x_cat[:, :d].cpu().double(), nf, ~st["navi_invalid"].cpu())
    h = O.mlp(P64, "add_latent.mlp", torch.cat([x2, zl.double()], 1), (0, 3, 6), True)
    x3 = h.masked_fill(st["latent_invalid"].cpu()[:, None], 0.0) + x2
    ref = torch.cat([O.mlp(P64, f"action_head.mlp_mean.{t}", x3, (0, 2, 4), False) for t in range(3)], 1)
    tol = 4e-3 * max(1.0, float(ref.abs().max()))
    errs = {}
    for chain in (True, False):
        m.opt["chain"] = chain
        lat = torch.cat([torch.zeros(M, d), zl], 1).to(DEV)
        navi = dict(pose=navi_pose, feat=feat, latent_cat=lat, latent_feat=True)
        n0 = ops.LAUNCHES
        act = m.heads(x_cat, st, navi)
        torch.cuda.synchronize()
        assert (ops.LAUNCHES - n0 == 2) == chain  # pose_emb + the chain program
        errs[chain] = float((act.cpu().double() - ref).abs().max())
        assert errs[chain] < tol, (chain, errs[chain], tol)
        assert float((lat[:, :d].cpu().double() - x2).abs().max()) < 4e-3 * max(1.0, float(x2.abs().max()))
        if chain:
            spec = m._heads_program().spec
            init = [x_cat.cpu(), ops.pose_emb(navi_pose, m.freq_rpe, d, frame=st["pose"], frame_div=1).cpu(),
                    feat.cpu(), st["navi_invalid"].cpu(), torch.cat([torch.zeros(M, d), zl], 1), st["latent_invalid"].cpu(),
                    torch.zeros(M, 6)]
            X, E, _ = CR.interpret(spec, init, torch.arange(M), bound=True)
            assert bool(((act.cpu().double() - X[6]).abs() <= E[6]).all())
            assert bool(((lat[:, :d].cpu().double() - X[4][:, :d]).abs() <= E[4][:, :d]).all())
            assert torch.equal(lat[:, d:].cpu(), init[4][:, d:])
    m.opt["chain"] = True
    print(f"\nheads vs float64 oracle: chain {errs[True]:.2e}, per layer {errs[False]:.2e} (tolerance {tol:.1e})")


def _ffn_run(offset=0.0):
    """_ffn_program on 1000 seeded rows; with `offset`, every residual row is shifted by +-offset. Returns
    (program, CPU inputs, device bindings after the run, row mask, LayerNorm gamma, LayerNorm beta)."""
    m, P, cfg = _model()
    d, M = cfg["hidden_dim"], 1000
    p, nxt = "mp_encoder.tf_mp2mp.layers.0", "mp_encoder.tf_mp2mp.layers.1.norm1"
    q = m._ffn_program(p, d, nxt)
    g = torch.Generator().manual_seed(23)
    mask = torch.rand(M, generator=g) < 0.3
    init = [torch.randn(M, d, generator=g).half(), torch.randn(M, d, generator=g), mask.to(torch.uint8),
            torch.full((M, d), 7.0), torch.zeros(M, d, dtype=torch.float16)]
    if offset:
        sign = torch.where(torch.rand(M, 1, generator=torch.Generator().manual_seed(29)) < 0.5, -1.0, 1.0)
        init[1] += offset * sign
    out = [t.to(DEV) for t in init]
    q.run(out, M)
    return q, init, out, mask, P[f"{nxt}.weight"], P[f"{nxt}.bias"]


def _check_ffn(q, init, out, mask, beta):
    M, d = init[1].shape
    X, E, _ = CR.interpret(q.spec, init, torch.arange(M), bound=True)
    for i in (3, 4):
        assert bool(((out[i].cpu().double() - X[i]).abs() <= E[i]).all()), i
    assert float(out[3][mask.to(DEV)].abs().max()) == 0.0
    assert torch.equal(out[4][mask.to(DEV)].cpu(), beta.half().expand(int(mask.sum()), d))


def test_engine_ffn_program_vs_interpreter():
    """_ffn_program (LN rows -> FFN-1 + ReLU, 4 hidden slices -> FFN-2 + residual + row mask -> fp32 rows + next
    LayerNorm) against the interpreter on its own spec; masked rows are 0 and their LayerNorm rows exactly fp16(beta)."""
    q, init, out, mask, _, beta = _ffn_run()
    _check_ffn(q, init, out, mask, beta)


def test_engine_ffn_program_layernorm_far_from_zero():
    """The FFN program with every residual row shifted by +-1000, so the LayerNorm sees rows whose mean is hundreds of
    times their spread: the interpreter check as above, and the fp16 LayerNorm rows against float64 LayerNorm of the
    program's own fp32 rows within tests/_linear_ref.ln_out_bound (group sums of depth 33). A one-pass
    E[v^2] - E[v]^2 loses the variance to cancellation here and misses that bound by orders of magnitude."""
    q, init, out, mask, gamma, beta = _ffn_run(1000.0)
    _check_ffn(q, init, out, mask, beta)
    y = out[3].cpu()
    ratio = float((y.double().mean(1).abs() / y.double().std(1).clamp_min(1e-30))[~mask].min())
    assert ratio > 100, ratio
    ref, _, _ = LR.layernorm_ref_f64(y, gamma, beta)
    bound = LR.ln_out_bound(y, gamma, beta, group_depth=33)
    err = (out[4].cpu().double() - ref).abs()
    r = float((err / bound).max())
    print(f"\nchain LayerNorm, mean / std >= {ratio:.0f}: worst ln_out error / bound {r:.3g}")
    assert r <= 1.0, f"{int((err > bound).sum())} ln_out values outside the bound, worst {r:.3g} x"


# ------------------------------------------------------------------------------------------------ refusals
def _cu(**kw):
    u = ops._ChainUnit()
    for f in ("mask_pre", "mask_post", "res", "out_buf", "out_g", "out_h", "ln_out", "src"):
        setattr(u, f, -1)
    for i in range(4):
        u.a_buf[i] = -1
    for k, v in kw.items():
        if k == "a_buf":
            for i, b in enumerate(v):
                u.a_buf[i] = b
        else:
            setattr(u, k, v)
    return u


def _encode(units, n_buf=4):
    blob = (ctypes.c_uint8 * L.load().tb_chain_program_bytes())()
    return L.load().tb_chain_encode((ops._ChainUnit * len(units))(*units), len(units), n_buf, blob)


def test_encoder_refusals():
    """One case for every refusal of tb_chain_encode, each with its code (n_units / n_buf: test_mlp_chain_cpu.py)."""
    w = torch.zeros(256, 512, dtype=torch.float16, device=DEV)
    b = torch.zeros(512, device=DEV)
    W = lambda K=128, N=128, off=0: dict(W=w.data_ptr() + off, K=K, N=N)  # noqa: E731
    ld = _cu(kind=1, src=0, lds=128, out_buf=0)
    gm = lambda **kw: _cu(**dict(dict(kind=0, a_buf=[0], out_buf=1, **W()), **kw))  # noqa: E731
    BAD, MIS, UNS = CR.TB_ERR_BAD_SHAPE, CR.TB_ERR_MISALIGNED, CR.TB_ERR_UNSUPPORTED
    assert _encode([ld, gm()]) == CR.TB_OK
    cases = [
        ([_cu(kind=1, src=0, lds=128, out_buf=4)], BAD),                              # out_buf >= n_buf
        ([ld, gm(out_buf=4)], BAD),
        ([_cu(kind=1, src=15, lds=128, out_buf=0)], BAD),                             # binding index 15
        ([ld, gm(out_g=15, ldg=128)], BAD), ([ld, gm(res=-2)], BAD), ([ld, gm(mask_pre=16)], BAD),
        ([_cu(kind=1, src=0, lds=128, out_buf=0, src_col=2)], BAD),                   # fp32 LOAD: 4-element multiples
        ([_cu(kind=1, src=0, lds=126, out_buf=0)], BAD),
        ([_cu(kind=1, src=0, lds=128, out_buf=0, src_col=4, src_f16=1)], BAD),        # fp16 LOAD: 8-element multiples
        ([_cu(kind=1, src=0, lds=132, out_buf=0, src_f16=1)], BAD),
        ([_cu(kind=1, src=0, lds=128)], BAD),                                         # LOAD without out_buf
        ([ld, gm(**W(K=96))], BAD), ([ld, gm(**W(K=576), a_buf=[0, 0, 0, 0])], BAD),  # K % 64, K > 512
        ([ld, gm(n0=128)], BAD), ([ld, gm(n_valid=129)], BAD), ([ld, gm(kind=2)], BAD),
        ([ld, gm(**W(off=2))], MIS), ([ld, gm(bias=b.data_ptr() + 4)], MIS),
        ([ld, gm(res=1, ldr=130)], MIS), ([ld, gm(res=1, ldr=128, res_col=2)], MIS),
        ([ld, gm(out_h=1, ldh=132)], MIS), ([ld, gm(out_h=1, ldh=128, h_col=4)], MIS),
        ([ld, gm(ln_out=1, ld_ln=132, ln_gamma=b.data_ptr(), ln_beta=b.data_ptr())], MIS),
        ([ld, gm(ln_out=1, ld_ln=128, ln_beta=b.data_ptr())], MIS),                   # ln_out without gamma
        ([ld, gm(ln_out=1, ld_ln=128, ln_gamma=b.data_ptr())], MIS),                  # ... or beta
        ([ld, gm(ln_out=1, ld_ln=128, ln_gamma=b.data_ptr() + 4, ln_beta=b.data_ptr())], MIS),
        ([ld, gm(a_buf=[1])], BAD),                                                   # reads a buffer nobody wrote
        ([ld, gm(**W(K=256), a_buf=[0, 2])], BAD),
        ([ld] + [gm(**W(K=64, N=128 + i)) for i in range(25)], UNS),                  # 25 distinct (W, K, N)
    ]
    for i, (units, code) in enumerate(cases):
        assert _encode(units) == code, (i, code)
    assert _encode([ld] + [gm(**W(K=64, N=128 + i)) for i in range(24)]) == CR.TB_OK
    # the same pointer with another K or N is another weight matrix (its own tensor map)
    same = [ld] + [gm(**W(K=64 * (1 + i % 2), N=128 + i // 2)) for i in range(31)]
    assert _encode(same) == UNS and _encode(same[:25]) == CR.TB_OK


def _runtime_program():
    """LOAD (binding 0, fp32) -> GEMM with mask_pre 1, residual 2, out_g 3 (vector path), out_h 4, ln_out 5."""
    w = torch.randn(128, 128, generator=torch.Generator().manual_seed(2)).half().to(DEV)
    gam, bet = torch.ones(128, device=DEV), torch.zeros(128, device=DEV)
    p = ops.ChainProgram(DEV, 2)
    p.load(0, 128, 0)
    p.gemm(w, [0], None, mask_pre=1, res=2, ldr=128, out_g=3, ldg=128, out_h=4, ldh=128, ln_out=5, ld_ln=128,
           ln_gamma=gam, ln_beta=bet)
    return p.finish()


def test_run_time_binding_refusals_launch_nothing():
    """tb_chain_run checks every binding the program uses before the launch: a short list, a NULL binding, each
    misaligned kind and a LOAD that reads what the launch writes are refused with their codes; nothing is launched and
    no output changes."""
    p = _runtime_program()
    M = 256
    big = torch.randn(M, 136, device=DEV)
    binds = [torch.randn(M, 128, device=DEV), torch.zeros(M, dtype=torch.uint8, device=DEV), torch.randn(M, 128, device=DEV),
             torch.full((M, 128), 3.0, device=DEV), torch.zeros(M, 128, dtype=torch.float16, device=DEV),
             torch.zeros(M, 128, dtype=torch.float16, device=DEV)]
    ptr = [t.data_ptr() for t in binds]
    snap = [t.clone() for t in binds]
    lib = L.load()

    def run(ptrs, n=None):
        arr = (ctypes.c_void_p * len(ptrs))(*ptrs)
        return lib.tb_chain_run(L.ptr(p.blob), p.host, arr, len(ptrs) if n is None else n, M, L.stream())

    cases = [(ptr[:5], CR.TB_ERR_BAD_SHAPE), (ptr[:1], CR.TB_ERR_BAD_SHAPE), (ptr, CR.TB_ERR_BAD_SHAPE, 4)]
    for k in range(6):
        cases.append((ptr[:k] + [None] + ptr[k + 1:], CR.TB_ERR_NULL))
    for k, off in ((0, 4), (2, 4), (3, 4), (3, 8), (4, 2), (4, 8), (5, 8)):  # LOAD, residual, out_g, out_h, ln_out
        cases.append((ptr[:k] + [big.data_ptr() + off] + ptr[k + 1:], CR.TB_ERR_MISALIGNED))
    for k in (3, 4, 5):                                                        # LOAD source written by the launch
        cases.append(([ptr[k]] + ptr[1:], CR.TB_ERR_UNSUPPORTED))
    n0 = ops.LAUNCHES
    for i, c in enumerate(cases):
        assert run(*c[:1], *c[2:]) == c[1], (i, c[1])
    torch.cuda.synchronize()
    assert ops.LAUNCHES == n0
    for a, b in zip(binds, snap):
        assert torch.equal(a, b)
    with pytest.raises(RuntimeError):
        p.run(binds[:5], M)
    assert run(ptr) == CR.TB_OK  # the valid bindings run
    torch.cuda.synchronize()
    assert not torch.equal(binds[3], snap[3])


def test_load_may_read_disjoint_columns_of_an_output():
    """The head chain's pattern: one LOAD reads the right half of a buffer whose left half a unit writes through out_g
    (same pitch, disjoint columns) - accepted and computed as the interpreter does; overlapping columns are refused."""
    w = torch.randn(128, 128, generator=torch.Generator().manual_seed(4)).half()
    M = 300
    for g_col, ok in ((0, True), (64, False)):
        spec = [CR._unit("load", src=0, lds=256, out_buf=0, src_col=128, f16=False),
                CR._unit("gemm", w=w, a_bufs=[0], out_g=0, ldg=256, g_col=g_col)]
        p = _build(spec, 2, {})
        init = [torch.randn(M, 256)]
        out = [init[0].to(DEV)]
        if ok:
            p.run(out, M)
            X, E, _ = CR.interpret(spec, init, torch.arange(M), bound=True)
            assert bool(((out[0].cpu().double() - X[0]).abs() <= E[0]).all())
            assert torch.equal(out[0][:, 128:].cpu(), init[0][:, 128:])
        else:
            with pytest.raises(RuntimeError):
                p.run(out, M)
            assert torch.equal(out[0].cpu(), init[0])


# ------------------------------------------------------------------------------------------------ out_h and n_valid
@pytest.mark.parametrize("n_valid", [1, 6, 31, 32, 33, 127])
def test_out_h_writes_only_n_valid_columns(n_valid):
    """out_h follows n_valid like out_g: columns h_col + c for c < n_valid only, with or without a buffer output
    (before the fix a unit without out_buf wrote whole 32-column slices: columns up to 31 at n_valid = 6)."""
    M = 200
    w = (torch.randn(128, 128, generator=torch.Generator().manual_seed(n_valid)) / 11).half()
    for out_buf in (-1, 1):
        spec = [CR._unit("load", src=0, lds=128, out_buf=0, src_col=0, f16=False),
                CR._unit("gemm", w=w, a_bufs=[0], out_buf=out_buf, out_h=1, ldh=280, h_col=8, n_valid=n_valid,
                         out_g=2, ldg=267, g_col=1)]
        init = [torch.randn(M, 128), torch.full((M, 280), CR.SENTINEL16, dtype=torch.int16).view(torch.float16),
                torch.full((M, 267), CR.SENTINEL32, dtype=torch.int32).view(torch.float32)]
        out = [t.to(DEV) for t in init]
        _build(spec, 2, {}).run(out, M)
        for i, c0 in ((1, 8), (2, 1)):
            got = out[i].cpu()
            assert torch.equal(_bits(got[:, :c0]), _bits(init[i][:, :c0]))
            assert torch.equal(_bits(got[:, c0 + n_valid:]), _bits(init[i][:, c0 + n_valid:])), (i, out_buf)
            assert not bool(torch.isnan(got[:, c0:c0 + n_valid].float()).any())


# ------------------------------------------------------------------------------------------------ fp16 range guard
def test_fp16_range_guard():
    """Values past 65504 saturate to exactly +-65504 (never inf) in buffers and out_h and set the tb_set_fp16_flag
    word; the same values leaving through fp32 out_g only, or in out_h columns past n_valid, do not."""
    M = 300
    flag = ops.fp16_flag(DEV)
    eye = (torch.eye(128) * 1000).half()
    x = torch.randn(M, 128, generator=torch.Generator().manual_seed(8)) * 0.01
    x[:, 3] = 100.0  # column 3: 1e5, past the fp16 range in every row
    x[:, 3][::2] = -100.0

    def run(spec, nb=3):
        init = [x, torch.zeros(M, 128, dtype=torch.float16), torch.zeros(M, 128)]
        out = [t.to(DEV) for t in init]
        flag.zero_()
        _build(spec, nb, {}).run(out, M)
        torch.cuda.synchronize()
        return int(flag.item()), out

    ld = CR._unit("load", src=0, lds=128, out_buf=0, src_col=0, f16=False)
    one = (torch.eye(128)).half()
    # out_h only
    f, out = run([ld, CR._unit("gemm", w=eye, a_bufs=[0], out_h=1, ldh=128)])
    assert f == 1 and torch.equal(out[1][:, 3].abs().float().cpu(), torch.full((M,), 65504.0))
    assert bool(torch.isfinite(out[1].float()).all())
    # through a buffer, read back by an identity unit
    f, out = run([ld, CR._unit("gemm", w=eye, a_bufs=[0], out_buf=1),
                  CR._unit("gemm", w=one, a_bufs=[1], out_g=2, ldg=128)])
    assert f == 1 and torch.equal(out[2][:, 3].cpu(), torch.where(x[:, 3] > 0, 65504.0, -65504.0))
    # fp32 out_g only: the full value, no flag
    f, out = run([ld, CR._unit("gemm", w=eye, a_bufs=[0], out_g=2, ldg=128)])
    assert f == 0 and float(out[2][:, 3].abs().min()) == 1e5
    # out_h with the large column past n_valid: not stored, no flag; inside n_valid: flag
    f, _ = run([ld, CR._unit("gemm", w=eye, a_bufs=[0], out_h=1, ldh=128, n_valid=3)])
    assert f == 0
    f, _ = run([ld, CR._unit("gemm", w=eye, a_bufs=[0], out_h=1, ldh=128, n_valid=4)])
    assert f == 1
    flag.zero_()
