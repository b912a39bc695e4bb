"""Host-side composition of the CUDA kernels into the reference's modules (eval mode, HPTR config).

Mirrors, function by function, the reference call chain (paths relative to the reference's src/):
  MapEncoder.forward             models/map_encoder.py:50-113
  TrafficLightEncoder.pre_compute / forward     models/traffic_light.py:76-154, 184-246
  AgentEncoder._forward_hptr     models/agent_encoder.py:114-178, 321-387
  TransformerRPE / AttentionRPE  models/modules/transformer_rpe.py:175-245, attention_rpe.py:58-198
  NaviEncoder / AddNaviLatent / ActionHead / TrafficLightStatePredictor
Weights arrive under the reference's state_dict names (params.param_shapes) and are re-packed once into the
fused projection matrices described in DESIGN.md §3 (exact re-association, done in float64).
All tensors here are 2-D [rows, channels] views of flat HBM buffers; every compute step is one ops.* launch.
"""
import math
from typing import Dict, Optional


import torch
from torch import Tensor

from . import ops

H = 4


def fuse_attention(P: Dict[str, Tensor], prefix: str, d: int, n_head: int = H, differentiable: bool = False
                   ) -> Dict[str, Tensor]:
    """attention_rpe.py:35-41,92-97,147-161,180-186 -> packed projections.
    in-proj rows: [ q*s (d) | u*s (H*d_rpe) | k (d) | v (d) ],  s = log2(e)/sqrt(d_head)
        u_h = W_rk,h^T q_h  =>  W_u[h] = W_rk,h^T W_q,h ,  b_u[h] = W_rk,h^T b_q,h
    out-proj columns: [ W_o (d) | W_o[:,h] W_rv,h (H*d_rpe) ],  bias b_o + W_o b_rv
    (the logit constant q_h.b_rk,h is softmax-invariant and dropped).
    `differentiable` (training path): the same re-packing with torch ops on the parameters' device, so autograd maps the
    gradients of the packed matrices back onto the reference's parameters (b_rk gets none: it cancels in the softmax)."""
    if differentiable:
        f64 = lambda k: P[f"{prefix}.{k}"].double()  # noqa: E731
    else:
        f64 = lambda k: P[f"{prefix}.{k}"].detach().double().cpu()  # noqa: E731
    w_in, b_in = f64("in_proj_weight"), f64("in_proj_bias")
    w_o, b_o = f64("out_proj_weight"), f64("out_proj_bias")
    w_r, b_r = f64("linear_rpe.weight"), f64("linear_rpe.bias")
    dh = d // n_head
    d_rpe = w_r.shape[1]
    s = math.log2(math.e) / math.sqrt(dh)
    w_q, b_q = w_in[:d] * s, b_in[:d] * s
    w_rk, w_rv, b_rv = w_r[:d], w_r[d:], b_r[d:]
    w_u, b_u, w_oz = [], [], []
    for h in range(n_head):
        sl = slice(h * dh, (h + 1) * dh)
        w_u.append(w_rk[sl].T @ w_q[sl])          # [d_rpe, d]
        b_u.append(w_rk[sl].T @ b_q[sl])          # [d_rpe]
        w_oz.append(w_o[:, sl] @ w_rv[sl])        # [d, d_rpe]
    w_qu = torch.cat([w_q] + w_u, 0)
    b_qu = torch.cat([b_q] + b_u, 0)
    out = dict(
        w_in_self=torch.cat([w_qu, w_in[d:]], 0), b_in_self=torch.cat([b_qu, b_in[d:]], 0),
        w_in_q=w_qu, b_in_q=b_qu, w_kv=w_in[d:], b_kv=b_in[d:],
        w_out=torch.cat([w_o] + w_oz, 1), b_out=b_o + w_o @ b_rv,
    )
    return {k: v.float().contiguous() for k, v in out.items()}


def head_interleave_perm(d: int = 128, n_head: int = H) -> Tensor:
    """Row order of a q / k / v projection block for tb_knarpe_attn flags bit 4: position
    64*(h>>1) + 16*(c>>3) + 8*(h&1) + (c&7) holds channel c of head h (d == 128, 4 heads of 32)."""
    assert d == 128 and n_head == 4
    s = torch.arange(d)
    head = 2 * (s >> 6) + ((s >> 3) & 1)
    return 32 * head + 8 * ((s >> 4) & 3) + (s & 7)


def _probe_fp32(fn):
    """Error-attribution hook of profiles/parity_probe.py: with `model._probe_heads_fp32` set, the decorated head
    functions run on the fp32 path while the rest of the model keeps its precision. Never set on the product path."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *a, **k):
        if getattr(self, "_probe_heads_fp32", False) and self.precision != 0:
            saved = (self.precision, self.kv_half)
            self.precision, self.kv_half = 0, False
            try:
                return fn(self, *a, **k)
            finally:
                self.precision, self.kv_half = saved
        return fn(self, *a, **k)
    return wrapped


class HotPathModel:
    """Device-resident weights + the kernel sequences of the hot-path modules."""

    # per-instance A/B switches of the tensor-core mode (defaults = the measured-best paths): head-interleaved q / K / V
    # rows, LayerNorm fused into the producing projection, head chain as one tb_chain_run program. Set before the first
    # forward (`model.opt["attn_il"] = False`); used by the bit-identity / equivalence tests and the profiling scripts.
    _OPT = dict(attn_il=True, ln_fused=True, chain=True)

    @property
    def opt(self) -> dict:
        if "_opt" not in self.__dict__:
            self._opt = dict(self._OPT)
        return self._opt

    def __init__(self, P: Dict[str, Tensor], cfg: dict, sizes: dict, device="cuda", precision: int = 0):
        self.cfg, self.sz, self.dev, self.precision = cfg, sizes, torch.device(device), precision
        self.d = cfg["hidden_dim"]
        self.kv_half = precision == 1 and self.d == 128  # fp16 K|V tables + tensor-core attention (tb_knarpe_attn bit 1)
        self.W = cfg["temp_window_size"]
        self.P = {k: v.detach().to(self.dev, torch.float32).contiguous() for k, v in P.items()}
        self.fa: Dict[str, Dict[str, Tensor]] = {}
        for k in P:
            if k.endswith(".in_proj_weight"):
                p = k[: -len(".in_proj_weight")]
                self.fa[p] = {n: t.to(self.dev) for n, t in fuse_attention(P, p, self.d).items()}
        self.freq_rpe = ops.pe_freq_xy(self.d, cfg["pose_rpe"]["theta_xy"], self.dev)          # d_rpe = hidden
        self.freq_ag = ops.pe_freq_xy(self.d // 2, cfg["ag_encoder"]["pose_emb"]["theta_xy"], self.dev)
        # action head: first layers of the 3 type branches stacked (action_head.py:25-36)
        self.act_w0 = torch.cat([self.P[f"action_head.mlp_mean.{t}.fc_layers.0.weight"] for t in range(3)], 0)
        self.act_b0 = torch.cat([self.P[f"action_head.mlp_mean.{t}.fc_layers.0.bias"] for t in range(3)], 0)
        self.act_w4 = torch.block_diag(*[self.P[f"action_head.mlp_mean.{t}.fc_layers.4.weight"] for t in range(3)]
                                       ).contiguous()
        self.act_b4 = torch.cat([self.P[f"action_head.mlp_mean.{t}.fc_layers.4.bias"] for t in range(3)], 0)

    @classmethod
    def from_state_dict(cls, sd: Dict[str, Tensor], d_model: int, theta_xy: float = 1e3, device="cuda",
                        precision: int = 0) -> "HotPathModel":
        """Runner over an arbitrary module's state_dict (used by the drop-in nn.Modules in reference_api.py)."""
        self = cls.__new__(cls)
        self.cfg, self.sz, self.dev, self.precision = None, None, torch.device(device), precision
        self.d, self.W = d_model, None
        self.kv_half = precision == 1 and d_model == 128
        self.P = {k: v.detach().to(self.dev, torch.float32).contiguous() for k, v in sd.items()}
        self.fa = {}
        for k in sd:
            if k.endswith("in_proj_weight"):
                p = k[: -len(".in_proj_weight")] if k.endswith(".in_proj_weight") else ""
                P = sd if p else {f".{n}": t for n, t in sd.items()}
                self.fa[p] = {n: t.to(self.dev) for n, t in fuse_attention(P, p, d_model).items()}
        self.freq_rpe = ops.pe_freq_xy(d_model, theta_xy, self.dev)
        return self

    # ------------------------------------------------------------------------------------------ helpers
    @property
    def gp(self) -> int:
        """tb_linear precision of the projections: in the strict-parity mode (precision 0) large projections run as
        3xTF32 on the tensor cores (fp32-class accuracy, ops.linear precision 3) unless `fp32_tc` is switched off."""
        return 3 if (self.precision == 0 and getattr(self, "fp32_tc", True)) else self.precision

    def lin(self, x, wname, relu=False, **kw):
        return ops.linear(x, self.P[f"{wname}.weight"], self.P[f"{wname}.bias"], relu=relu, precision=self.gp,
                          **kw)

    def ln(self, x, name, half: bool = False):
        """LayerNorm; `half`: fp16 rows for a following kind::f16 projection (tensor-core mode)."""
        return ops.layernorm(x, self.P[f"{name}.weight"], self.P[f"{name}.bias"],
                             out_dtype=torch.float16 if half else torch.float32)

    @property
    def kv_il(self) -> bool:
        """Head-interleaved q / K / V rows (tb_knarpe_attn flags bit 4): every attention of the tensor-core mode runs
        on the pair kernel, so the projections write the layout it gathers with 256-bit loads."""
        return self.kv_half and self.opt["attn_il"]

    def _proj(self, x: Tensor, key: str, w: Tensor, b: Tensor, il_blocks=(), **kw):
        """Projection of LayerNorm output: fp16 rows x fp16 weights (tb_linear precision 2) or the fp32 / tf32 path.
        `il_blocks`: first rows of the d-row blocks (q, k, v) stored head-interleaved when kv_il is on."""
        if x.dtype == torch.float16:
            if il_blocks and self.kv_il:
                w, b = self._interleaved(key, w, b, il_blocks)
                key += ".il"
            return ops.linear(x, self._half(key, w), b, precision=2, **kw)
        return ops.linear(x, w, b, precision=self.gp, **kw)

    def _interleaved(self, key: str, w: Tensor, b: Tensor, blocks):
        if not hasattr(self, "_w_il"):
            self._w_il = {}
        if key not in self._w_il:
            rows = torch.arange(w.shape[0], device=w.device)
            perm = head_interleave_perm(self.d).to(w.device)
            for r0 in blocks:
                rows[r0:r0 + self.d] = r0 + perm
            self._w_il[key] = (w[rows].contiguous(), b[rows].contiguous())
        return self._w_il[key]

    def mlp(self, x, prefix, idxs, end_act, **last_kw):
        for n, i in enumerate(idxs):
            last = n == len(idxs) - 1
            x = self.lin(x, f"{prefix}.fc_layers.{i}", relu=(not last) or end_act, **(last_kw if last else {}))
        return x

    def pointnet(self, x: Tensor, row_invalid: Tensor, G: int, Lg: int, prefix: str) -> Tensor:
        """polyline_encoder.py:50-53 + pooling.py:18-19,38. x [G*L, d]."""
        # De-duplicated form: cat(h, max_g) W^T = h W_left^T + (max_g W_right^T), the second term being one row per
        # group -> a [G, d/2] GEMM whose result enters the big GEMM as a grouped bias. Rows stay d/2 wide, the
        # broadcast copy of the max is never written, and the final token is [max h | max h]. Values on invalid rows
        # differ from the reference's (zeros) but are masked out of every max, exactly like there.
        half = self.d // 2
        h = self.lin(x, f"{prefix}.mlp_layers.0.fc_layers.0", relu=True)
        for i in (1, 2):
            m = ops.pointnet_pool(h, row_invalid, G, Lg, 1)
            w_l, w_r = self._pointnet_split(prefix, i)
            gb = ops.linear(m, w_r, self.P[f"{prefix}.mlp_layers.{i}.fc_layers.0.bias"], precision=self.gp)
            h = ops.linear(h, w_l, gb, relu=True, bias_group=Lg, precision=self.gp)
        return ops.pointnet_pool(h, row_invalid, G, Lg, 2)

    def _pointnet_split(self, prefix: str, i: int):
        key = f"{prefix}.{i}"
        if not hasattr(self, "_pn_split"):
            self._pn_split = {}
        if key not in self._pn_split:
            w = self.P[f"{prefix}.mlp_layers.{i}.fc_layers.0.weight"]
            half = w.shape[1] // 2
            self._pn_split[key] = (w[:, :half].contiguous(), w[:, half:].contiguous())
        return self._pn_split[key]

    def kv_table(self, feat: Tensor, layer_prefix: str, norm: str, attn: str = "attn", out: Optional[Tensor] = None
                 ) -> Tensor:
        """K/V rows of a target table for one layer: W_kv LN(x) + b  (project-once-then-gather, DESIGN.md §3)."""
        f = self.fa[f"{layer_prefix}.{attn}"]
        x = self.ln(feat, f"{layer_prefix}.{norm}", half=self.kv_half)
        if self.kv_half:  # tensor-core mode: fp16 tables straight from the projection's epilogue
            tbl = out if out is not None else torch.empty(x.shape[0], 2 * self.d, dtype=torch.float16, device=x.device)
            self._proj(x, f"{layer_prefix}.{attn}.w_kv", f["w_kv"], f["b_kv"], out_h=tbl, col_h=0,
                       il_blocks=(0, self.d))
            return tbl
        return ops.linear(x, f["w_kv"], f["b_kv"], precision=self.gp, out=out)

    def _in_self(self, f, x, K, key=""):
        """[q|u] and the token's own [k|v] rows from one projection: one fp16 [q|u|k|v] row buffer in tensor-core mode
        (the pair attention kernel's operands), one fp32 buffer otherwise."""
        nq = self.d + H * self.d
        if self.kv_half:
            row = torch.empty(x.shape[0], nq + 2 * self.d, dtype=torch.float16, device=x.device)
            self._proj(x, f"{key}.w_in_self", f["w_in_self"], f["b_in_self"], out_h=row, col_h=0,
                       il_blocks=(0, nq, nq + self.d))
            return row[:, :nq], row[:, nq:]
        proj = ops.linear(x, f["w_in_self"], f["b_in_self"], precision=self.gp)
        return proj, proj[:, nq:]

    def _in_q(self, f, x, key=""):
        """[q|u] rows for a cross-attention: fp16 in tensor-core mode (the attention kernel's MMA operands)."""
        if self.kv_half:
            qu = torch.empty(x.shape[0], self.d + H * self.d, dtype=torch.float16, device=x.device)
            self._proj(x, f"{key}.w_in_q", f["w_in_q"], f["b_in_q"], out_h=qu, col_h=0, il_blocks=(0,))
            return qu
        return ops.linear(x, f["w_in_q"], f["b_in_q"], precision=self.gp)

    def _attend(self, fa, proj, B, S, kv0, T0, div0, K0, knn, kv1=None, T1=0, div1=1, K1=0):
        d = self.d
        if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (proj, kv0, kv1)):
            from . import autograd as AG  # training path: differentiable core (tb_knarpe_attn_bwd)
            return AG.knarpe_attn(proj[:, :d + H * d], kv0, T0, div0, K0, knn["idx"], knn["inv"], knn["rel"],
                                  self.freq_rpe, B, S, d, H, kv1=kv1, T1=T1, div1=div1, K1=K1,
                                  fast_trig=self.precision == 1)
        return ops.knarpe_attn(proj[:, :d], proj[:, d:d + H * d], kv0, T0, div0, K0, knn["idx"], knn["inv"],
                               knn.get("rel"), self.freq_rpe, B, S, d, H, kv1=kv1, T1=T1, div1=div1, K1=K1,
                               emb=knn.get("emb"), fast_trig=self.precision == 1, interleaved=self.kv_il,
                               out_dtype=torch.float16 if self.kv_half else torch.float32)

    def _half(self, key: str, w: Tensor) -> Tensor:
        """fp16 copy of a weight matrix (tensor-core mode: operands of the kind::f16 projections), made once."""
        if not hasattr(self, "_w_half"):
            self._w_half = {}
        if key not in self._w_half:
            self._w_half[key] = w.to(torch.float16).contiguous()
        return self._w_half[key]

    @property
    def chain_fused(self) -> bool:
        """Head chain as one fused tcgen05 chain program (tb_chain_run) in the tensor-core mode; `opt["chain"] = False`
        keeps the one-launch-per-layer path (A/B and bisecting)."""
        return self.opt["chain"]

    def _ffn_program(self, p: str, ldy: int, ln_next: Optional[str]):
        """bindings: 0 LayerNorm rows fp16 [M,d], 1 residual fp32 [M,d], 2 row mask u8 [M], 3 out fp32 (ld ldy),
        4 LayerNorm rows of the result fp16 [M,d] (when ln_next)."""
        if not hasattr(self, "_chain"):
            self._chain = {}
        key = ("ffn", p, ldy, ln_next)
        if key not in self._chain:
            d = self.d
            w1 = self._half(f"{p}.linear1", self.P[f"{p}.linear1.weight"])
            w2 = self._half(f"{p}.linear2", self.P[f"{p}.linear2.weight"])
            nh = w1.shape[0] // d
            assert w1.shape == (nh * d, d) and w2.shape == (d, nh * d) and nh <= 4
            q = ops.ChainProgram(self.dev, n_buf=nh)
            q.load(0, d, 0, f16=True)
            # hidden slice t -> buffer t + 1; the last one overwrites the input buffer (its MMAs, and those of the earlier
            # slices, have read it by the time its epilogue runs): nh buffers leave a deeper weight ring than nh + 1
            hb = [(t + 1) % nh for t in range(nh)]
            for t in range(nh):
                q.gemm(w1, [0], self.P[f"{p}.linear1.bias"], n0=t * d, relu=True, out_buf=hb[t])
            ln = dict(ln_out=4, ld_ln=d, ln_gamma=self.P[f"{ln_next}.weight"], ln_beta=self.P[f"{ln_next}.bias"]) if ln_next else {}
            q.gemm(w2, hb, self.P[f"{p}.linear2.bias"], res=1, ldr=d, mask_post=2, out_g=3, ldg=ldy, **ln)
            self._chain[key] = q.finish()
        return self._chain[key]

    def _heads_program(self):
        """The per-step head chain as one program. bindings: 0 x_cat fp32 [M,2d] (agent feature in the left half),
        1 PoseEmb of the destination in the agent frame fp32 [M,d], 2 static navigation feature fp32 [M,d],
        3 navi_invalid u8 [M], 4 latent cat buffer fp32 [M,2d] (left: add_navi result, written here; right: static latent
        feature), 5 latent_invalid u8 [M], 6 act_branch fp32 [M,6]."""
        if not hasattr(self, "_chain"):
            self._chain = {}
        if "heads" not in self._chain:
            self._chain["heads"] = self._heads_chain().finish()
        return self._chain["heads"]

    def _heads_chain(self, half: bool = True):
        """The units of `_heads_program`, not encoded. half=False keeps the fp32 weights: a description only, for a
        float64 reference of the same program (tests/_chain_ref.py)."""
        d = self.d
        hw = (lambda n: self._half(n, self.P[f"{n}.weight"])) if half else (lambda n: self.P[f"{n}.weight"])  # noqa: E731
        b = lambda n: self.P[f"{n}.bias"]  # noqa: E731
        q = ops.ChainProgram(self.dev, n_buf=4)
        q.load(1, d, 1)                                                                        # pe -> B1
        q.load(0, 2 * d, 0)                                                                    # x -> B0 (used by add_navi.mlp)
        n = "navi_encoder.mlp_pe.fc_layers.0"
        q.gemm(hw(n), [1], b(n), res=2, ldr=d, out_buf=2)                                      # nf (navigation.py:73-79)
        for i, (src_b, dst_b) in zip((0, 3, 6), ((2, 1), (1, 2), (2, 1))):                     # add_navi.mlp_in
            n = f"add_navi.mlp_in.fc_layers.{i}"
            q.gemm(hw(n), [src_b], b(n), relu=True, out_buf=dst_b, mask_post=3 if i == 6 else -1)
        n = "add_navi.mlp.fc_layers.0"
        q.gemm(hw(n), [0, 1], b(n), relu=True, out_buf=2)                                      # cat(x, a1)
        n = "add_navi.mlp.fc_layers.3"
        q.gemm(hw(n), [2], b(n), relu=True, out_buf=3)
        n = "add_navi.mlp.fc_layers.6"
        q.gemm(hw(n), [3], b(n), relu=True, mask_pre=3, res=0, ldr=2 * d, out_buf=0, out_g=4, ldg=2 * d)  # x2
        q.load(4, 2 * d, 1, src_col=d)                                                         # latent feature -> B1
        n = "add_latent.mlp.fc_layers.0"
        q.gemm(hw(n), [0, 1], b(n), relu=True, out_buf=2)
        n = "add_latent.mlp.fc_layers.3"
        q.gemm(hw(n), [2], b(n), relu=True, out_buf=3)
        n = "add_latent.mlp.fc_layers.6"
        q.gemm(hw(n), [3], b(n), relu=True, mask_pre=5, res=4, ldr=2 * d, out_buf=0)           # x3
        w0 = self._half("action_head.w0", self.act_w0) if half else self.act_w0
        for t in range(3):                                                                     # action_head.py:78-82
            q.gemm(w0, [0], self.act_b0, n0=t * d, relu=True, out_buf=1 + t)
        for t in range(3):
            n = f"action_head.mlp_mean.{t}.fc_layers.2"
            q.gemm(hw(n), [1 + t], b(n), relu=True, out_buf=1 + t)
        w4 = self._half("action_head.w4", self.act_w4) if half else self.act_w4
        q.gemm(w4, [1, 2, 3], self.act_b4, out_g=6, ldg=6, n_valid=6)
        return q

    @property
    def ln_fused(self) -> bool:
        """LayerNorm of the residual stream inside the epilogue of the projection that produces it (tb_linear_ln)."""
        return self.kv_half and self.d == 128 and self.opt["ln_fused"]

    def _out_proj(self, p: str, f: dict, o: Tensor, nv: Tensor, res: Tensor, ln_next: Optional[str] = None):
        """Output projection over [ov|z] (fp16 rows in tensor-core mode -> kind::f16 MMA, fp32 accumulate/residual).
        `ln_next`: name of the LayerNorm applied to the result next -> returns (result, fp16 LN rows) from one launch."""
        if o.dtype == torch.float16:
            w = self._half(f"{p}.w_out", f["w_out"])
            if ln_next is not None and self.ln_fused:
                return ops.linear_ln(o, w, f["b_out"], self.P[f"{ln_next}.weight"], self.P[f"{ln_next}.bias"], mask_pre=nv,
                                     res=res, precision=2)
            y = ops.linear(o, w, f["b_out"], mask_pre=nv, res=res, precision=2)
        else:
            y = ops.linear(o, f["w_out"], f["b_out"], mask_pre=nv, res=res, precision=self.gp)
        return y if ln_next is None else (y, self.ln(y, ln_next, half=self.kv_half))

    def tf_layer(self, p: str, mode: str, src: Tensor, src_inv: Tensor, B: int, S: int, knn_self: dict,
                 cross: Optional[dict] = None, out: Optional[Tensor] = None, before_self=None, before_cross=None,
                 ln_in: Optional[Tensor] = None, ln_next: Optional[str] = None):
        """TransformerRPE.forward (transformer_rpe.py:175-245), eval mode. `before_self` / `before_cross` are join
        hooks called right before the self / cross attention launch (streams that produce the neighbour lists).
        `ln_in`: the layer's first LayerNorm already applied to `src` (by the previous layer's epilogue);
        `ln_next`: name of the LayerNorm the caller applies to the result next -> returns (result, LN rows)."""
        d, pr = self.d, self.precision
        if mode == "dec_cross_attn":
            f = self.fa[f"{p}.attn_src"]
            x0 = ln_in if ln_in is not None else self.ln(src, f"{p}.norm_src", half=self.kv_half)
            proj, kv = self._in_self(f, x0, knn_self["idx"].shape[-1], f"{p}.attn_src")
            if before_self is not None:
                before_self()
            o, nv = self._attend(f, proj, B, S, kv, S, 1, knn_self["idx"].shape[-1], knn_self)
            src, x1 = self._out_proj(f"{p}.attn_src", f, o, nv, src, ln_next=f"{p}.norm1")
            f = self.fa[f"{p}.attn"]
            proj = self._in_q(f, x1, f"{p}.attn")
            if before_cross is not None:
                before_cross()
            o, nv = self._attend(f, proj, B, S, cross["kv0"], cross["T0"], cross["div0"], cross["K0"], cross,
                                 cross.get("kv1"), cross.get("T1", 0), cross.get("div1", 1), cross.get("K1", 0))
            src, x2 = self._out_proj(f"{p}.attn", f, o, nv, src, ln_next=f"{p}.norm2")
        else:  # enc_self_attn: q and k/v both from norm1(src) (:218-221)
            f = self.fa[f"{p}.attn"]
            x0 = ln_in if ln_in is not None else self.ln(src, f"{p}.norm1", half=self.kv_half)
            proj, kv = self._in_self(f, x0, knn_self["idx"].shape[-1], f"{p}.attn")
            o, nv = self._attend(f, proj, B, S, kv, S, 1, knn_self["idx"].shape[-1], knn_self)
            src, x2 = self._out_proj(f"{p}.attn", f, o, nv, src, ln_next=f"{p}.norm2")
        # (A fused FFN-1 -> ReLU -> FFN-2 chain program exists - `_ffn_program`, profiles/chain_probe.py - but measured
        # slower than the two launches at 65,536 rows (83 vs 58 us, profiles/r2_notes.md 3); it is not on this path.)
        if self.kv_half:  # FFN hidden (ReLU output) as fp16: written by the first projection, read by a kind::f16 one
            h = torch.empty(x2.shape[0], self.P[f"{p}.linear1.weight"].shape[0], dtype=torch.float16, device=x2.device)
            self._proj(x2, f"{p}.linear1", self.P[f"{p}.linear1.weight"], self.P[f"{p}.linear1.bias"], relu=True, out_h=h,
                       col_h=0)
            w2 = self._half(f"{p}.linear2", self.P[f"{p}.linear2.weight"])
            if ln_next is not None and self.ln_fused:  # the next layer's first LayerNorm rides on this epilogue
                return ops.linear_ln(h, w2, self.P[f"{p}.linear2.bias"], self.P[f"{ln_next}.weight"],
                                     self.P[f"{ln_next}.bias"], res=src, mask_post=src_inv, out=out, precision=2)
            y = ops.linear(h, w2, self.P[f"{p}.linear2.bias"], res=src, mask_post=src_inv, out=out, precision=2)
        else:
            h = self.lin(x2, f"{p}.linear1", relu=True)
            y = self.lin(h, f"{p}.linear2", res=src, mask_post=src_inv, out=out)
        return y if ln_next is None else (y, self.ln(y, ln_next, half=self.kv_half))

    def tf_stack(self, prefix: str, n_layer: int, mode: str, tok: Tensor, layer_kw, ln_in: Optional[Tensor] = None
                 ) -> Tensor:
        """n_layer TransformerRPE layers; layer i's closing projection also produces layer i+1's first LayerNorm rows
        (tb_linear_ln) when the tensor-core mode allows it. `layer_kw(i)` -> (positional args after src, kwargs)."""
        first = "norm_src" if mode == "dec_cross_attn" else "norm1"
        for i in range(n_layer):
            args, kw = layer_kw(i)
            nxt = f"{prefix}.{i + 1}.{first}" if (i + 1 < n_layer and self.ln_fused) else None
            r = self.tf_layer(f"{prefix}.{i}", mode, tok, *args, ln_in=ln_in, ln_next=nxt, **kw)
            tok, ln_in = r if nxt is not None else (r, None)
        return tok

    # ------------------------------------------------------------------------------------------ map (once / scene)
    def map_encoder(self, mp_valid: Tensor, mp_attr: Tensor, mp_pose: Tensor) -> Dict[str, Tensor]:
        """MapEncoder.forward, map_encoder.py:50-113. The geometric front-end (polyline-local frame + 7 features,
        :65-77, pose_emb.py:59-89) runs once per scene and is plain torch; MLP / PointNet / KNN / 8 KNARPE layers
        are the CUDA kernels."""
        d, sz = self.d, self.sz
        n_sc, n_mp, Ln = mp_valid.shape
        tok_pose = mp_pose[:, :, 0].contiguous()
        tok_inv = ~mp_valid[:, :, 0]
        c, s = torch.cos(tok_pose[..., 2]), torch.sin(tok_pose[..., 2])
        rot = torch.stack([torch.stack([c, -s], -1), torch.stack([s, c], -1)], -2)
        xy = torch.matmul(mp_pose[..., :2] - tok_pose[:, :, None, :2], rot)
        yaw = mp_pose[..., 2] - tok_pose[..., 2:3]
        pe7 = _encode_polyline(xy, torch.stack([yaw.cos(), yaw.sin()], -1))
        attr = torch.cat([mp_attr[:, :, None, :].expand(-1, -1, Ln, -1),
                          torch.eye(Ln, device=self.dev)[None, None].expand(n_sc, n_mp, -1, -1)], -1)
        M = n_sc * n_mp * Ln
        x = torch.empty(M, d, device=self.dev)
        x[:, d - 7:] = pe7.reshape(M, 7)
        self.mlp(attr.reshape(M, -1).contiguous(), "mp_encoder.input_encoder.mlp", (0, 2, 4), False, out=x[:, : d - 7])
        tok = self.pointnet(x, (~mp_valid).reshape(-1).contiguous(), n_sc * n_mp, Ln, "mp_encoder.pl_encoder")
        idx, inv, rel = ops.knn_select(tok_pose, tok_inv, tok_pose, tok_inv, sz["k_mp2mp"], sz["dl_mp"])
        knn = dict(idx=idx, inv=inv, rel=rel)
        flat_inv = tok_inv.reshape(-1).contiguous()
        tok = self.tf_stack("mp_encoder.tf_mp2mp.layers", self.cfg["mp_encoder"]["n_layer_tf"], "enc_self_attn", tok,
                            lambda i: ((flat_inv, n_sc, n_mp, knn), {}))
        return dict(mp_token_invalid=tok_inv.contiguous(), mp_token_feature=tok.view(n_sc, n_mp, d),
                    mp_token_pose=tok_pose, knn_mp2mp=knn, **self.sorted_map(tok_pose, tok_inv))

    @staticmethod
    def sorted_map(tok_pose: Tensor, tok_inv: Tensor) -> Dict[str, Tensor]:
        """x-sorted copy of the (static) map token poses for the per-step agent -> map select (tb_knn_select row_state)."""
        order = torch.argsort(tok_pose[..., 0], dim=1)
        return dict(mp_sorted_pose=torch.gather(tok_pose, 1, order[..., None].expand(-1, -1, 3)).contiguous(),
                    mp_sorted_invalid=torch.gather(tok_inv, 1, order).contiguous(),
                    mp_sorted_index=order.to(torch.int32).contiguous())

    # ------------------------------------------------------------------------------------------ traffic lights
    def tl_pre_compute(self, tl_valid: Tensor, tl_attr: Tensor, tl_pose: Tensor, mp: Dict[str, Tensor]) -> dict:
        """TrafficLightEncoder.pre_compute, traffic_light.py:76-154 + per-layer map K/V tables of tf_tl2tlmp."""
        sz, d = self.sz, self.d
        n_sc, n_tl = tl_valid.shape
        n_mp = mp["mp_token_pose"].shape[1]
        inv = (~tl_valid).contiguous()
        tl_pose = tl_pose.contiguous()
        feat2d = mp["mp_token_feature"].reshape(n_sc * n_mp, d)
        attr = ops.gather_rows(mp["mp_token_feature"].contiguous(), tl_attr.to(torch.int32).reshape(-1).contiguous(),
                               n_tl)                                                              # :115
        i1, m1, r1 = ops.knn_select(tl_pose, inv, tl_pose, inv, sz["k_tl2tl"], sz["dl_tl"])       # :119,129-135
        i2, m2, r2 = ops.knn_select(tl_pose, inv, mp["mp_token_pose"], mp["mp_token_invalid"], sz["k_tl2mp"],
                                    sz["dl_tl"])                                                  # :120-145
        kv = [self.kv_table(feat2d, f"tl_encoder.tf_tl2tlmp.layers.{i}", "norm_tgt")
              for i in range(self.cfg["tl_encoder"]["n_layer_tf"])]
        W = self.W
        return dict(tl_token_invalid=inv, tl_token_pose=tl_pose, tl_token_attr=attr,
                    tl_attr_rows=attr.view(n_sc * n_tl, 1, d).expand(-1, W, -1).reshape(-1, d).contiguous(),
                    knn_self=dict(idx=i1, inv=m1, rel=r1),
                    cross=[dict(kv0=kv[i], T0=n_mp, div0=1, K0=sz["k_tl2mp"], idx=i2, inv=m2, rel=r2)
                           for i in range(len(kv))], n_sc=n_sc, n_tl=n_tl)

    def tl_forward(self, hist_tl: Tensor, d_step: Tensor, tl: dict, out_feat: Optional[Tensor] = None,
                   out_logits: Optional[Tensor] = None, with_logits: bool = True):
        """TrafficLightEncoder.forward (traffic_light.py:210-240) + TrafficLightStatePredictor (:270-286, pre-clamp).
        hist_tl [Bt, n_tl, W, 5] u8 ring. `with_logits=False`: tokens only (the latent encoders' TL branch)."""
        from . import lib as L
        Bt, n_tl, W, d = tl["n_sc"], tl["n_tl"], self.W, self.d
        M = Bt * n_tl * W
        attr = torch.empty(M, 5 + W, device=self.dev)
        row_inv = torch.empty(M, dtype=torch.bool, device=self.dev)
        # d_step: the shared loop counter, or (training: all steps of a rollout as one batch) one counter per batch row
        L.check(L.load().tb_tl_featurize_ex(L.ptr(hist_tl), L.ptr(ops._u8(tl["tl_token_invalid"])), L.ptr(d_step),
                                            1 if d_step.numel() > 1 else 0, Bt, n_tl, W, L.ptr(attr), 5 + W,
                                            L.ptr(ops._u8(row_inv)), L.stream()), "tb_tl_featurize_ex")
        ops._count()
        x = self.mlp(attr, "tl_encoder.input_encoder.mlp", (0, 2, 4), False, res=tl["tl_attr_rows"])  # :176-180
        tok = self.pointnet(x, row_inv, Bt * n_tl, W, "tl_encoder.temp_encoder")                      # :228
        flat_inv = tl["tl_token_invalid"].reshape(-1)
        nl = self.cfg["tl_encoder"]["n_layer_tf"]
        tok = self.tf_stack("tl_encoder.tf_tl2tlmp.layers", nl, "dec_cross_attn", tok,                  # :231-240
                            lambda i: ((flat_inv, Bt, n_tl, tl["knn_self"], tl["cross"][i]),
                                       dict(out=out_feat if i == nl - 1 else None)))
        if not with_logits:
            return tok, None
        # training: the state predictor reads detached tokens (traffic_light.py:279-280, detach_tl_feature)
        tok_in = tok.detach() if getattr(self, "detach_tl_feature", False) else tok
        logits = self.mlp(tok_in, "tl_state_predictor.mlp", (0, 2, 4), False, out=out_logits)         # :284
        return tok, logits

    # ------------------------------------------------------------------------------------------ agents (per step)
    def ag_static(self, mp: Dict[str, Tensor]) -> list:
        """Per-scene map K/V tables of the 4 tf_ag2agmptl layers (static: shared by all rollouts and steps)."""
        n_sc, n_mp, d = mp["mp_token_feature"].shape
        feat2d = mp["mp_token_feature"].reshape(n_sc * n_mp, d)
        return [self.kv_table(feat2d, f"ag_encoder.tf_ag2agmptl.layers.{i}", "norm_tgt")
                for i in range(self.cfg["ag_encoder"]["n_layer_tf"])]

    def ag_forward(self, st: dict, mp: Dict[str, Tensor], kv_mp: list, tl: dict, tl_feat: Tensor, R: int,
                   out: Optional[Tensor] = None, aux: Optional[dict] = None, before_tl=None, knn_stream=None,
                   knn_stream2=None, kv_tl: Optional[list] = None, tl_pose_div: Optional[int] = None) -> Tensor:
        """AgentEncoder._forward_hptr (agent_encoder.py:114-178). `st` holds the rollout state rings
        (engine.RolloutState); batch b uses map / traffic-light tables of scene b // R. `kv_tl`: per-layer K|V tables
        of the traffic-light tokens when the caller already built them (on the TL stream); `before_tl` is then
        only called right before the first cross-attention instead of before layer 0. `tl_pose_div`: batch rows per row
        of tl["tl_token_pose"] when that differs from the rows per TL table (training: per-scene poses, per-step tables);
        `st["d_step"]` may hold one loop counter per batch row (tb_ag_featurize_ex)."""
        from . import lib as L
        sz, d, W = self.sz, self.d, self.W
        B, A = st["B"], st["A"]
        n_mp, n_tl = mp["mp_token_pose"].shape[1], tl["n_tl"]
        tl_div = B // (tl_feat.shape[0] // n_tl)  # rollout-scenes per traffic-light batch row (R if TL runs per scene)
        M, MW = B * A, B * A * W
        tok_pose = torch.empty(B, A, 3, device=self.dev)
        tok_inv = torch.empty(B, A, dtype=torch.bool, device=self.dev)
        fused = self.kv_half and W <= 16 and d == 128  # tensor-core mode: one fused kernel for the history encoder
        hist = (L.ptr(st["hist_valid"]), L.ptr(st["hist_pose"]), L.ptr(st["hist_motion"]), L.ptr(st["ag_attr"]),
                L.ptr(st["d_step"]), L.ptr(self.freq_ag), B, A, W)
        per_row_step = st["d_step"].numel() > 1
        stride = 1 if per_row_step else 0
        if fused:  # token pose / validity first (tiny), so that the KNN selects start beside the fused encoder
            L.check(L.load().tb_ag_featurize_ex(*hist[:5], stride, *hist[5:], L.ptr(tok_pose), L.ptr(ops._u8(tok_inv)),
                                                None, None, 0, None, 0, L.stream()), "tb_ag_featurize_ex")
        else:
            row_inv = torch.empty(MW, dtype=torch.bool, device=self.dev)
            attr = torch.empty(MW, 9 + W, device=self.dev)
            x = torch.empty(MW, d, device=self.dev)
            L.check(L.load().tb_ag_featurize_ex(*hist[:5], stride, *hist[5:], L.ptr(tok_pose),
                                                L.ptr(ops._u8(tok_inv)), L.ptr(ops._u8(row_inv)), L.ptr(attr), 9 + W,
                                                L.ptr(x[:, d // 2:]), d, L.stream()), "tb_ag_featurize_ex")
        ops._count()
        # re-localisation + KNN re-selection, every step (:321-387). The three selects only need the token poses, so
        # they run on a forked stream beside the (bandwidth-bound) input MLP + PointNet projections.
        Kc, Ka = sz["k_ag2mp"] + sz["k_ag2tl"], sz["k_ag2ag"]
        i_aa = torch.empty(B, A, Ka, dtype=torch.int32, device=self.dev)
        m_aa = torch.empty(B, A, Ka, dtype=torch.bool, device=self.dev)
        r_aa = torch.empty(B, A, Ka, 3, device=self.dev)
        cidx = torch.empty(B, A, Kc, dtype=torch.int32, device=self.dev)
        cinv = torch.empty(B, A, Kc, dtype=torch.bool, device=self.dev)
        crel = torch.empty(B, A, Kc, 3, device=self.dev)

        def select_self():
            ops.knn_select(tok_pose, tok_inv, tok_pose, tok_inv, Ka, sz["dl_ag"], out=(i_aa, m_aa, r_aa))

        def select_cross():
            if "knn_state" in st and "mp_sorted_pose" in mp:  # static targets + per-row state: x-slab fast path
                ops.knn_select(tok_pose, tok_inv, mp["mp_sorted_pose"], mp["mp_sorted_invalid"], sz["k_ag2mp"],
                               sz["dl_ag"], tgt_div=R, out=(cidx, cinv, crel), koff=0,
                               index_map=mp["mp_sorted_index"], row_state=st["knn_state"], sorted_by_x=True)
            else:
                ops.knn_select(tok_pose, tok_inv, mp["mp_token_pose"], mp["mp_token_invalid"], sz["k_ag2mp"],
                               sz["dl_ag"], tgt_div=R, out=(cidx, cinv, crel), koff=0)
            ops.knn_select(tok_pose, tok_inv, tl["tl_token_pose"], tl["tl_token_invalid"], sz["k_ag2tl"], sz["dl_ag"],
                           tgt_div=tl_pose_div or tl_div, out=(cidx, cinv, crel), koff=sz["k_ag2mp"],
                           row_state=st.get("knn_state_tl"))  # static targets too: bracketed bisection

        # The agent->agent list is needed by the first self-attention, the agent->map/TL lists only by the first
        # cross-attention: with two side streams the big map select also overlaps layer 0's projections + self-attn.
        main = torch.cuda.current_stream()
        join_self = join_cross = None
        if knn_stream is not None:
            s2 = knn_stream2 if knn_stream2 is not None else knn_stream
            s2.wait_stream(main)
            with torch.cuda.stream(s2):
                select_self()
            knn_stream.wait_stream(main)
            with torch.cuda.stream(knn_stream):
                select_cross()
            join_self = lambda: main.wait_stream(s2)          # noqa: E731
            join_cross = lambda: main.wait_stream(knn_stream)  # noqa: E731
        if fused:
            blob, bias = self._ag_frontend_weights()
            tok = torch.empty(M, d, device=self.dev)
            tp2, ti2 = torch.empty_like(tok_pose), torch.empty_like(tok_inv)  # same values as tok_pose / tok_inv
            ln0 = None
            if self.ln_fused:  # the first LayerNorm of the agent transformer rides on the encoder's epilogue
                ln0 = torch.empty(M, d, dtype=torch.float16, device=self.dev)
                nm = "ag_encoder.tf_ag2agmptl.layers.0.norm_src"
                ln_args = (L.ptr(self.P[f"{nm}.weight"]), L.ptr(self.P[f"{nm}.bias"]), L.ptr(ln0), d)
            else:
                ln_args = (None, None, None, 0)
            L.check(L.load().tb_ag_frontend_ex(*hist[:5], stride, *hist[5:], L.ptr(blob), L.ptr(bias), L.ptr(tok), d,
                                               L.ptr(tp2), L.ptr(ops._u8(ti2)), *ln_args, L.stream()),
                    "tb_ag_frontend_ex")                                                              # :130-162
            ops._count()
        else:
            ln0 = None
            self.mlp(attr, "ag_encoder.input_encoder.mlp", (0, 2, 4), False, out=x[:, : d // 2])      # :159
            tok = self.pointnet(x, row_inv, M, W, "ag_encoder.temp_encoder")                          # :162
        if knn_stream is None:
            select_self()
            select_cross()
        knn_self = dict(idx=i_aa, inv=m_aa, rel=r_aa)
        flat_inv = tok_inv.reshape(-1)
        nl = self.cfg["ag_encoder"]["n_layer_tf"]
        if aux is not None:
            aux.update(tok_pose=tok_pose, tok_inv=tok_inv, tok0=tok, knn_self=knn_self, cidx=cidx, cinv=cinv, crel=crel)
        if before_tl is not None and kv_tl is None:
            before_tl()  # join point: the traffic-light branch (side stream) must have produced tl_feat

        def join_first_cross():  # the first consumer of the agent->map/TL lists and of the TL tables
            if join_cross is not None:
                join_cross()
            if before_tl is not None and kv_tl is not None:
                before_tl()

        def layer_kw(i):
            p = f"ag_encoder.tf_ag2agmptl.layers.{i}"
            kv1 = kv_tl[i] if kv_tl is not None else self.kv_table(tl_feat, p, "norm_tgt")
            cross = dict(kv0=kv_mp[i], T0=n_mp, div0=R, K0=sz["k_ag2mp"], kv1=kv1, T1=n_tl, div1=tl_div,
                         K1=sz["k_ag2tl"], idx=cidx, inv=cinv, rel=crel)
            return (flat_inv, B, A, knn_self, cross), dict(out=out if i == nl - 1 else None,
                                                           before_self=join_self if i == 0 else None,
                                                           before_cross=join_first_cross if i == 0 else None)

        tok = self.tf_stack("ag_encoder.tf_ag2agmptl.layers", nl, "dec_cross_attn", tok, layer_kw, ln_in=ln0)
        return tok

    def ag_tl_tables(self, tl_feat: Tensor, out: Optional[list] = None) -> list:
        """K|V tables of the traffic-light tokens for the 4 agent layers (rows of tf_ag2agmptl's cross-attention)."""
        return [self.kv_table(tl_feat, f"ag_encoder.tf_ag2agmptl.layers.{i}", "norm_tgt",
                              out=out[i] if out is not None else None)
                for i in range(self.cfg["ag_encoder"]["n_layer_tf"])]

    # ------------------------------------------------------------------------------------------ destinations (once / scene)
    def navi_predictor(self, ag_valid: Tensor, ag_attr: Tensor, ag_motion: Tensor, ag_pose: Tensor,
                       mp: Dict[str, Tensor], ag_type: Tensor, mp_type: Tensor, scene_chunk: int = 4) -> Tensor:
        """NaviPredictor.forward, "dest" mode (navigation.py:175-278; SURVEY 8(f) rank 3): destination logits
        [n_sc, n_ag, n_mp] — the once-per-scene step right before the rollout loop (waymo_motion.py:469-495).
        The first Linear of the pair MLP over [agent | polyline | PE(rel pose)] is split column-wise: the agent part
        is one row per agent and enters as a grouped bias, so the [n_sc, n_ag, n_mp, 384] input is never built."""
        d, W = self.d, self.W
        n_sc, A, n_step = ag_valid.shape
        if n_step > W:                                                                                   # :210-214
            # the token pose uses the full history (:204) - identical here because the last valid step is kept
            ag_valid, ag_motion, ag_pose, n_step = ag_valid[:, :, -W:], ag_motion[:, :, -W:], ag_pose[:, :, -W:], W
        tok_valid = ag_valid.any(-1)
        last = n_step - 1 - torch.max(ag_valid.flip(2).to(torch.uint8), dim=2)[1]
        tok_pose = torch.gather(ag_pose, 2, last[:, :, None, None].expand(-1, -1, 1, 3)).squeeze(2)
        tok_pose = tok_pose.masked_fill(~tok_valid[..., None], 0.0).contiguous()                         # :204
        M, MW = n_sc * A, n_sc * A * n_step
        attr = torch.cat([ag_attr[:, :, None, :].expand(-1, -1, n_step, -1), ag_motion,
                          torch.eye(W, device=self.dev)[None, None, -n_step:].expand(n_sc, A, -1, -1)], -1)  # :221-228
        x = torch.empty(MW, d, device=self.dev)
        self.mlp(attr.reshape(MW, -1).contiguous(), "navi_predictor.input_encoder.mlp", (0, 2, 4), False,
                 out=x[:, : d // 2])
        ops.pose_emb(ag_pose.reshape(MW, 3), self.freq_ag, d // 2, frame=tok_pose, frame_div=n_step, out=x[:, d // 2:])
        tok = self.pointnet(x, (~ag_valid).reshape(-1).contiguous(), M, n_step, "navi_predictor.temp_encoder")  # :232
        pr = "navi_predictor.mlp.fc_layers"
        w0 = self.P[f"{pr}.0.weight"]
        a_part = ops.linear(tok, w0[:, :d].contiguous(), self.P[f"{pr}.0.bias"], precision=self.gp)
        w_mr = w0[:, d:].contiguous()
        n_mp = mp["mp_token_pose"].shape[1]
        logits = torch.empty(n_sc, A, n_mp, device=self.dev)
        for s0 in range(0, n_sc, scene_chunk):
            ns = min(scene_chunk, n_sc - s0)
            Pn = ns * A * n_mp
            X = torch.empty(Pn, 2 * d, device=self.dev)
            X[:, :d].view(ns, A, n_mp, d).copy_(mp["mp_token_feature"][s0:s0 + ns, None])
            pose_rows = mp["mp_token_pose"][s0:s0 + ns, None].expand(-1, A, -1, -1).reshape(Pn, 3)
            ops.pose_emb(pose_rows, self.freq_rpe, d, frame=tok_pose[s0:s0 + ns], frame_div=n_mp, out=X[:, d:])  # :259-260
            h = ops.linear(X, w_mr, a_part[s0 * A:(s0 + ns) * A], bias_group=n_mp, precision=self.gp)
            h = ops.layernorm(h, self.P[f"{pr}.1.weight"], self.P[f"{pr}.1.bias"], relu=True, out=h)      # mlp.py:47-51
            h = self.lin(h, f"{pr}.3")
            h = ops.layernorm(h, self.P[f"{pr}.4.weight"], self.P[f"{pr}.4.bias"], relu=True, out=h)
            logits[s0:s0 + ns] = self.lin(h, f"{pr}.6").view(ns, A, n_mp)
        # type masks (:265-278)
        mp_mask = mp["mp_token_invalid"] | ~(mp_type[:, :, :5].any(-1))
        inv = (mp_mask.unsqueeze(1) | (ag_type[:, :, [0]] & mp_type[:, :, 3].unsqueeze(1))
               | (ag_type[:, :, [1]] & mp_type[:, :, :4].any(-1).unsqueeze(1))
               | (ag_type[:, :, [2]] & mp_type[:, :, :3].any(-1).unsqueeze(1)))
        logits = logits.masked_fill(inv, float("-inf"))
        return logits.masked_fill((~tok_valid).unsqueeze(-1) | inv.all(-1, keepdim=True), 0.0)

    def _ag_frontend_weights(self):
        """fp16 weight blob + fp32 biases of tb_ag_frontend (layout: include/tb_knarpe.h), built once."""
        if not hasattr(self, "_ag_front"):
            from . import lib as L
            n = L.load().tb_ag_frontend_blob_halves()
            blob = torch.zeros(n, dtype=torch.float16, device=self.dev)
            names = [f"ag_encoder.input_encoder.mlp.fc_layers.{i}" for i in (0, 2, 4)] + \
                    [f"ag_encoder.temp_encoder.mlp_layers.{i}.fc_layers.0" for i in range(3)]
            off = 0
            for nm, stride in zip(names, (40, 72, 72, 136, 136, 136)):
                w = self.P[f"{nm}.weight"]
                assert w.shape[0] == 64 and w.shape[1] <= stride - 8, w.shape
                blob[off:off + 64 * stride].view(64, stride)[:, : w.shape[1]] = w.to(torch.float16)
                off += 64 * stride
            assert off == n
            bias = torch.cat([self.P[f"{nm}.bias"] for nm in names]).contiguous()
            self._ag_front = (blob, bias)
        return self._ag_front

    # ------------------------------------------------------------------------------------------ heads (per step)
    @_probe_fp32
    def navi_static(self, mp: Dict[str, Tensor], dest_idx: Tensor, R: int) -> dict:
        """Static halves of NaviEncoder.forward (navigation.py:65-71): mlp_mp(map feature of the destination) and the
        destination's global pose. dest_idx int32 [B, A]."""
        B, A = dest_idx.shape
        flat = dest_idx.reshape(-1).contiguous()
        f = ops.gather_rows(mp["mp_token_feature"].contiguous(), flat, A, R)
        pose = ops.gather_rows(mp["mp_token_pose"].contiguous(), flat, A, R)
        return dict(feat=self.lin(f, "navi_encoder.mlp_mp.fc_layers.0"), pose=pose)

    @_probe_fp32
    def latent_static(self, navi: dict, st: dict) -> None:
        """AddNaviLatent.mlp_in(latent) (add_navi_latent.py:50) depends only on the rollout's fixed latent sample:
        evaluated once per rollout into the right half of a persistent cat buffer."""
        d = self.d
        M = st["latent"].shape[0]
        cat = torch.zeros(M, 2 * d, device=self.dev)
        self.mlp(st["latent"], "add_latent.mlp_in", (0, 3, 6), True, mask_post=st["latent_invalid"].reshape(-1),
                 out=cat[:, d:])
        navi["latent_cat"] = cat
        navi["latent_feat"] = True

    @_probe_fp32
    def heads(self, x_cat: Tensor, st: dict, navi: dict) -> Tensor:
        """navi_encoder (per-step half) -> add_navi -> add_latent -> action-head branches
        (traffic_bots.py:191-217). x_cat [M, 2d] with the agent feature already in the left half.
        Returns act_branch [M, 6] (veh, ped, cyc) x (acc, yaw-rate) pre-tanh, unmasked."""
        d = self.d
        M = x_cat.shape[0]
        pe = ops.pose_emb(navi["pose"], self.freq_rpe, d, frame=st["pose"], frame_div=1)             # navigation.py:73-79
        if self.kv_half and self.chain_fused and d == 128 and "latent_cat" in navi and x_cat.is_contiguous():
            act = torch.empty(M, 6, device=self.dev)
            self._heads_program().run([x_cat, pe, navi["feat"], ops._u8(st["navi_invalid"]).reshape(-1), navi["latent_cat"],
                                       ops._u8(st["latent_invalid"]).reshape(-1), act], M)
            return act
        nf = self.lin(pe, "navi_encoder.mlp_pe.fc_layers.0", res=navi["feat"])
        # add_navi writes its result straight into the left half of add_latent's cat buffer
        x_cat2 = navi["latent_cat"] if "latent_cat" in navi else torch.empty(M, 2 * d, device=self.dev)
        for prefix, z, zinv, cat_in, cat_out in (("add_navi", nf, st["navi_invalid"], x_cat, x_cat2[:, :d]),
                                                 ("add_latent", st["latent"], st["latent_invalid"], x_cat2, None)):
            zinv = zinv.reshape(-1)                                                                  # add_navi_latent.py:46-64
            if prefix == "add_latent" and "latent_feat" in navi:
                # the latent sample is fixed for the whole rollout: mlp_in(latent) was evaluated once (latent_static)
                cat_in = navi["latent_cat"]
            else:
                self.mlp(z, f"{prefix}.mlp_in", (0, 3, 6), True, mask_post=zinv, out=cat_in[:, d:])
            h = self.mlp(cat_in, f"{prefix}.mlp", (0, 3, 6), True, mask_pre=zinv, res=cat_in[:, :d], out=cat_out)
        if self.kv_half:  # tensor-core mode: the two hidden layers of the 3 type branches as fp16 rows
            h0 = torch.empty(M, 3 * d, dtype=torch.float16, device=self.dev)
            ops.linear(h, self.act_w0, self.act_b0, relu=True, precision=1, out_h=h0, col_h=0)       # action_head.py:78-82
            h1 = torch.empty_like(h0)
            for t in range(3):
                nm = f"action_head.mlp_mean.{t}.fc_layers.2"
                ops.linear(h0[:, t * d:(t + 1) * d], self._half(nm, self.P[f"{nm}.weight"]), self.P[f"{nm}.bias"],
                           relu=True, precision=2, out_h=h1[:, t * d:(t + 1) * d], col_h=0)
            return ops.linear(h1, self._half("action_head.w4", self.act_w4), self.act_b4, precision=2)
        h0 = ops.linear(h, self.act_w0, self.act_b0, relu=True, precision=self.gp)            # action_head.py:78-82
        h1 = torch.empty_like(h0)
        for t in range(3):
            self.lin(h0[:, t * d:(t + 1) * d], f"action_head.mlp_mean.{t}.fc_layers.2", relu=True,
                     out=h1[:, t * d:(t + 1) * d])
        # last layers of the 3 type branches as ONE block-diagonal [6, 3d] projection of the stacked hidden rows
        return ops.linear(h1, self.act_w4, self.act_b4, precision=self.gp)


def _encode_polyline(pos: Tensor, dirv: Tensor) -> Tensor:
    """PoseEmb mode mpa_pl, utils/pose_emb.py:59-89 (once per scene)."""
    eps = torch.finfo(pos.dtype).eps
    proj = (-pos * dirv).sum(-1) / ((dirv * dirv).sum(-1) + eps)
    closest = pos + proj.clamp(0, 1).unsqueeze(-1) * dirv
    r = torch.norm(closest, dim=-1, keepdim=True)
    dn = torch.norm(dirv, dim=-1, keepdim=True)
    return torch.cat([r, closest / (r + eps), dirv / (dn + eps), dn,
                      torch.norm(pos + dirv - closest, dim=-1, keepdim=True)], -1)
