"""CPU: the fused MLP chain's float64 reference (tests/_chain_ref.py) against the oracle's head chain, the encoder's
rules on every generated program, the weight-ring depths, and the encoder's shape codes from the compiled library."""
import ctypes

import pytest
import torch

import _chain_ref as CR
from oracle import tb_oracle as O
from trafficbotsv1_5_b200 import config, lib, params


@pytest.fixture(scope="module")
def handle():
    lib.build()
    return lib.load()


def test_ring_depth_table():
    """Weight stages per (n_buf, unit count): (227 KB - 1 KB - 32 KB n_buf - 704 n_units - 4928) / 16 KB, capped at 8.
    6 buffers leave a single stage even for one unit, which is why the encoder accepts 2..5 only."""
    assert CR.tail_bytes(1) == 704 + 4928 and CR.tail_bytes(32) == 704 * 32 + 4928
    want = {2: (8, 8), 3: (7, 6), 4: (5, 4), 5: (3, 2)}
    for n_buf, (lo, hi) in want.items():
        for n in range(1, 33):
            assert CR.ring_depth(n_buf, n) == (lo if n <= 19 else hi), (n_buf, n)
    assert max(CR.ring_depth(6, n) for n in range(1, 33)) == 1
    # no unit count in 1..32 makes the 5-buffer ring shallower than 2: the encoder's n_stage < 2 refusal is unreachable
    assert min(CR.ring_depth(5, n) for n in range(1, 33)) == 2


def test_generated_programs_follow_encoder_rules():
    """Every generated program is one the encoder accepts (rules re-derived in Python), writes every global element
    from one unit only (the residual alias reads an earlier out_g at the same columns), and together the programs reach
    every ring depth 2..8, n_buf 2..5 and every epilogue flag."""
    depths, bufs, flags, n_valid, ks = set(), set(), set(), set(), set()
    most_waits = 0
    for seed, n_buf, n_units, long_run in CR.PROGRAMS:
        spec, nb = CR.gen_program(seed, n_buf, n_units, long_run)
        r = CR.encode_rules(spec, nb)
        assert r["code"] == CR.TB_OK, (seed, r)
        depths.add(r["n_stage"])
        bufs.add(nb)
        most_waits = max(most_waits, max(len(w) for w in r["waits"]))
        slots = []
        for s in spec:
            if s["kind"] == "load":
                flags.add("load16" if s["f16"] else "load32")
                if s["src_col"] > 0:
                    flags.add("src_col")
                continue
            ks.add(s["w"].shape[1])
            if s["relu"]:
                flags.add("relu")
            if s["bias"] is not None:
                flags.add("bias")
            for f in ("mask_pre", "mask_post", "res", "out_buf", "out_g", "out_h", "ln_out"):
                if s[f] >= 0:
                    flags.add(f)
            if s["res"] == 5:
                flags.add("res_alias")
                assert s["res_col"] in slots
            if s["out_g"] >= 0:
                flags.add("og_vector" if s["out_g"] == 5 else "og_scalar")
                if s["out_g"] == 5:
                    slots.append(s["g_col"])
            if s["out_g"] >= 0 or s["out_h"] >= 0:
                n_valid.add(s["n_valid"])
            if s["out_buf"] >= 0 and s["out_buf"] in s["a_bufs"]:
                flags.add("in_place")
            if len(set(s["a_bufs"])) < len(s["a_bufs"]):
                flags.add("same_buffer_twice")
            if s["n0"] > 0:
                flags.add("n0")
            if s["w"].shape[0] - s["n0"] < 128:
                flags.add("zero_fill_rows")
        outs = [(s["out_g"], s["g_col"]) for s in spec if s["kind"] == "gemm" and s["out_g"] >= 0]
        outs += [(s["out_h"], s["h_col"]) for s in spec if s["kind"] == "gemm" and s["out_h"] >= 0]
        assert len(outs) == len(set(outs)), "one writer per output slot"
    assert depths == set(range(2, 9)), depths
    assert bufs == {2, 3, 4, 5}
    assert ks == {64 * i for i in range(1, 9)}
    assert set(CR.N_VALID) <= n_valid, n_valid
    assert {"load16", "load32", "src_col", "relu", "bias", "mask_pre", "mask_post", "res", "res_alias", "out_buf", "og_vector",
            "og_scalar", "out_h", "ln_out", "in_place", "same_buffer_twice", "n0", "zero_fill_rows"} <= flags, flags
    # the most waits a unit can have: its (at most 4) input buffers' last writers + the GEMM 4 earlier
    spec, nb = CR.max_wait_program()
    r = CR.encode_rules(spec, nb)
    assert r["code"] == CR.TB_OK and max(len(w) for w in r["waits"]) == 5
    assert most_waits <= 5


def test_encoder_shape_codes_without_gpu(handle):
    """tb_chain_encode checks NULL, n_units and n_buf before it queries the driver; tb_chain_run its scalar arguments
    before it reads the program."""
    from trafficbotsv1_5_b200 import ops
    blob = (ctypes.c_uint8 * handle.tb_chain_program_bytes())()
    units = (ops._ChainUnit * 33)()
    enc = handle.tb_chain_encode
    assert enc(None, 1, 4, blob) == CR.TB_ERR_NULL
    assert enc(units, 1, 4, None) == CR.TB_ERR_NULL
    for n_units, n_buf in ((0, 4), (33, 4), (1, 1), (1, 6), (1, 7), (32, 6)):
        assert enc(units, n_units, n_buf, blob) == CR.TB_ERR_BAD_SHAPE, (n_units, n_buf)
    run = handle.tb_chain_run
    ptrs = (ctypes.c_void_p * 1)(None)
    assert run(None, blob, ptrs, 1, 4, None) == CR.TB_ERR_NULL
    assert run(128, blob, None, 1, 4, None) == CR.TB_ERR_NULL
    assert run(128, blob, ptrs, 1, 0, None) == CR.TB_ERR_BAD_SHAPE
    assert run(128, blob, ptrs, 16, 4, None) == CR.TB_ERR_BAD_SHAPE
    assert run(64, blob, ptrs, 1, 4, None) == CR.TB_ERR_MISALIGNED
    assert run(128, blob, ptrs, 1, 4, None) == CR.TB_ERR_BAD_SHAPE  # a zeroed blob: no units


def test_interpreter_heads_spec_matches_oracle():
    """The head chain as the engine builds it (HotPathModel._heads_chain with fp32 weights), run by the float64
    interpreter without fp16 rounding, is the oracle's navi_encoder.mlp_pe -> add_navi_latent x 2 -> the three
    action-head branches. Only float64 summation order differs (1e-10 relative)."""
    from trafficbotsv1_5_b200.model import HotPathModel
    cfg = config.default_model_cfg()
    P = params.init_params(cfg, 0)
    m = HotPathModel(P, cfg, config.derived_sizes(cfg), device="cpu", precision=1)
    spec = m._heads_chain(half=False).spec
    d, M = cfg["hidden_dim"], 300
    g = torch.Generator().manual_seed(3)
    x, pe, feat = (torch.randn(M, d, generator=g) for _ in range(3))
    z = torch.randn(M, P["add_latent.mlp_in.fc_layers.0.weight"].shape[1], generator=g)
    navi_inv, lat_inv = torch.rand(M, generator=g) < 0.2, torch.rand(M, generator=g) < 0.2
    P64 = {k: v.double() for k, v in P.items()}
    zl = O.mlp(P64, "add_latent.mlp_in", z.double(), (0, 3, 6), True).masked_fill(lat_inv[:, None], 0.0)
    x_cat = torch.cat([x, torch.zeros(M, d)], 1)
    lat_cat = torch.cat([torch.zeros(M, d, dtype=torch.float64), zl], 1)
    bind = [x_cat, pe, feat, navi_inv.to(torch.uint8), lat_cat, lat_inv.to(torch.uint8), torch.zeros(M, 6)]
    X, _, _ = CR.interpret(spec, bind, torch.arange(M), round16=False)
    nf = feat.double() + O.mlp(P64, "navi_encoder.mlp_pe", pe.double(), (0,), False)
    x2 = O.add_navi_latent(P64, "add_navi", x.double(), nf, ~navi_inv)
    x3 = O.add_navi_latent(P64, "add_latent", x2, z.double(), ~lat_inv)
    act = torch.cat([O.mlp(P64, f"action_head.mlp_mean.{t}", x3, (0, 2, 4), False) for t in range(3)], 1)
    tol = 1e-10 * (1 + act.abs().max())
    assert float((X[6] - act).abs().max()) < tol
    assert float((X[4][:, :d] - x2).abs().max()) < 1e-10 * (1 + x2.abs().max())  # add_navi result, written by out_g
    assert torch.equal(X[4][:, d:], lat_cat[:, d:])                                 # the LOAD half is untouched


class _UnitDev(ctypes.Structure):
    """The device unit record of mlp_chain.cu (192 bytes at offset 64 of the host blob), for hand-made programs."""
    _fields_ = [(f, ctypes.c_int) for f in ("flags", "tmem_col", "out_off", "n_valid", "map", "n0", "nk", "n_wait")] + \
        [("wait", ctypes.c_int * 8), ("a_off", ctypes.c_int * 8)] + \
        [(f, ctypes.c_void_p) for f in ("bias", "ln_g", "ln_b")] + \
        [(f, ctypes.c_int) for f in ("mask_pre", "mask_post", "res", "ldr", "res_col", "out_g", "ldg", "g_col", "out_h",
                                     "ldh", "h_col", "ln_out", "ld_ln", "src", "lds", "src_col", "pad0", "pad1")]


F_LOAD, F_MPRE, F_RES, F_OG, F_OH, F_LN = 1, 4, 16, 64, 128, 256


def test_run_time_binding_refusals_without_gpu(handle):
    """tb_chain_run checks, from the host blob and before anything touches the device, every binding the program uses:
    index < n_bind, not NULL, aligned for its accesses, and no LOAD source that the launch writes. A hand-made program
    (LOAD 0 -> GEMM with mask_pre 1, residual 2, out_g 3, out_h 4, ln_out 5) with fake addresses: every case here is
    refused, so nothing is launched (an accepted case would launch; there is none)."""
    assert ctypes.sizeof(_UnitDev) == 192
    blob = (ctypes.c_uint8 * handle.tb_chain_program_bytes())()
    struct_hdr = (ctypes.c_int * 4).from_buffer(blob)
    struct_hdr[0], struct_hdr[2], struct_hdr[3] = 2, 2, 8
    units = (_UnitDev * 2).from_buffer(blob, 64)
    units[0].flags, units[0].src, units[0].lds = F_LOAD, 0, 128
    g = units[1]
    g.flags, g.n_valid, g.nk = F_MPRE | F_RES | F_OG | F_OH | F_LN, 128, 2
    g.mask_pre, g.res, g.ldr, g.out_g, g.ldg, g.out_h, g.ldh, g.ln_out, g.ld_ln = 1, 2, 128, 3, 128, 4, 128, 5, 128
    ptr = [1 << 20, (1 << 20) + 4096 + 1, 2 << 20, 3 << 20, 4 << 20, 5 << 20]  # the mask needs no alignment
    prog = 6 << 20

    def run(p, n=None):
        arr = (ctypes.c_void_p * max(len(p), 1))(*p)
        return handle.tb_chain_run(prog, blob, arr, len(p) if n is None else n, 256, None)

    assert run(ptr[:5]) == CR.TB_ERR_BAD_SHAPE and run(ptr[:1]) == CR.TB_ERR_BAD_SHAPE
    assert run(ptr, 4) == CR.TB_ERR_BAD_SHAPE
    for k in range(6):
        assert run(ptr[:k] + [None] + ptr[k + 1:]) == CR.TB_ERR_NULL, k
    for k, off in ((0, 4), (0, 8), (2, 4), (3, 4), (3, 8), (4, 2), (4, 8), (5, 8)):
        assert run(ptr[:k] + [ptr[k] + off] + ptr[k + 1:]) == CR.TB_ERR_MISALIGNED, (k, off)
    for k in (3, 4, 5):  # the LOAD reads what out_g / out_h / ln_out write
        assert run([ptr[k]] + ptr[1:]) == CR.TB_ERR_UNSUPPORTED, k
    g.ldg, g.g_col = 129, 1  # scalar out_g path: 4-byte rows
    assert run(ptr[:3] + [ptr[3] + 2] + ptr[4:]) == CR.TB_ERR_MISALIGNED
    # half-overlapping columns of the same pitch are refused too (the disjoint case runs on the GPU)
    g.ldg, g.g_col, g.n_valid = 256, 0, 128
    units[0].lds, units[0].src_col = 256, 64
    assert run([ptr[3]] + ptr[1:]) == CR.TB_ERR_UNSUPPORTED
    struct_hdr[0] = 33
    assert run(ptr) == CR.TB_ERR_BAD_SHAPE
