"""Tensor-level wrappers over the C ABI (include/tb_knarpe.h). torch is used for device memory and streams
only; every op below is one launch of a hand-written sm_100a kernel on torch's current stream."""
import ctypes
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import lib as L

LAUNCHES = 0  # number of kernels launched through this module (bench.py reports it as gpu_launches)


_FP16_FLAG = {}


def fp16_flag(device) -> Tensor:
    """The sticky fp16-saturation word of this process' device (tb_set_fp16_flag): allocated once, never freed (its
    address is baked into captured graphs), zeroed by the caller before a rollout and read after it."""
    dev = torch.device(device)
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _FP16_FLAG:
        assert not _FP16_FLAG, "one process drives one GPU (the flag pointer is a per-process setting)"
        _FP16_FLAG[key] = torch.zeros(1, dtype=torch.int32, device=dev)
        L.check(L.load().tb_set_fp16_flag(L.ptr(_FP16_FLAG[key])), "tb_set_fp16_flag")
    return _FP16_FLAG[key]


def _count(n=1):
    global LAUNCHES
    LAUNCHES += n


def _u8(t: Optional[Tensor]) -> Optional[Tensor]:
    if t is None:
        return None
    if t.dtype == torch.bool:
        return t.view(torch.uint8)
    assert t.dtype == torch.uint8, t.dtype
    return t


def _f32c(t: Tensor) -> Tensor:
    assert t.dtype == torch.float32 and t.is_cuda, (t.dtype, t.device)
    return t if t.is_contiguous() else t.contiguous()


def pe_freq_xy(pe_dim: int, theta: float = 1e3, device="cuda") -> Tensor:
    """PositionalEmbedding(dim=pe_dim/4, theta).freqs[::2] with the reference's own fp32 formula
    (utils/positional_emb.py:11): pe_dim/8 frequencies."""
    dim = pe_dim // 4
    f = 1.0 / (theta ** (torch.arange(0, dim, 2)[: dim // 2].float() / dim))
    return f.to(device)


def knn_select(src_pose: Tensor, src_invalid: Tensor, tgt_pose: Tensor, tgt_invalid: Tensor, k: int,
               dist_limit: float, tgt_div: int = 1, out: Optional[Tuple[Tensor, Tensor, Tensor]] = None,
               koff: int = 0, index_map: Optional[Tensor] = None, row_state: Optional[Tensor] = None,
               sorted_by_x: bool = False, reference: bool = False) -> Tuple[Tensor, Tensor, Tensor]:
    """Fused get_rel_pose + get_tgt_knn_idx (utils/rpe.py:9-90). Returns idx int32 [B,S,K], invalid bool [B,S,K],
    rel [B,S,K,3]; with `out`/`koff` writes into columns koff..koff+K of preallocated [B,S,ldk(,3)] buffers.
    reference=True runs the previous select kernels (TB_KNN_REFERENCE): the same lists and row states, bit for bit."""
    B, S, _ = src_pose.shape
    T = tgt_pose.shape[1]
    assert tgt_pose.shape[0] * tgt_div == B, (tgt_pose.shape, tgt_div, B)
    src_pose, tgt_pose = _f32c(src_pose), _f32c(tgt_pose)
    si, ti = _u8(src_invalid).contiguous(), _u8(tgt_invalid).contiguous()
    if out is None:
        idx = torch.empty(B, S, k, dtype=torch.int32, device=src_pose.device)
        inv = torch.empty(B, S, k, dtype=torch.bool, device=src_pose.device)
        rel = torch.empty(B, S, k, 3, dtype=torch.float32, device=src_pose.device)
    else:
        idx, inv, rel = out
    ldk = idx.shape[2]
    if index_map is not None:
        assert index_map.dtype == torch.int32 and index_map.is_contiguous() and index_map.shape == tgt_pose.shape[:2]
    if row_state is not None:
        assert row_state.dtype == torch.float32 and row_state.is_contiguous() and row_state.shape == (B, S, 3)
    L.check(L.load().tb_knn_select(L.ptr(src_pose), L.ptr(si), L.ptr(tgt_pose), L.ptr(ti), B, S, T, tgt_div, k,
                                   float(dist_limit), L.ptr(idx), L.ptr(_u8(inv)), L.ptr(rel), ldk, koff,
                                   L.ptr(index_map), L.ptr(row_state), int(sorted_by_x) | (2 if reference else 0), L.stream()),
            "tb_knn_select")
    _count()
    return idx, inv, rel


def knarpe_attn(q: Tensor, u: Tensor, kv0: Tensor, T0: int, div0: int, K0: int, idx: Tensor, invalid: Tensor,
                rel: Optional[Tensor], freq_xy: Tensor, B: int, S: int, D: int, H: int = 4,
                kv1: Optional[Tensor] = None, T1: int = 0, div1: int = 1, K1: int = 0,
                emb: Optional[Tensor] = None, out: Optional[Tensor] = None, fast_trig: bool = False,
                interleaved: bool = False,
                out_dtype: torch.dtype = torch.float32) -> Tuple[Tensor, Tensor]:
    """KNARPE core. q/u/kv*: 2-D (possibly column-sliced, row-strided) views; returns (out [B*S, D+H*D] = [ov|z],
    none_valid bool [B*S]). float16 kv tables select the tensor-core kernel (tb_knarpe_attn flags bit 1), a float16
    `out` (or out_dtype) the fp16 output rows (bit 2)."""
    M = B * S
    rpe_mma = kv0.dtype == torch.float16
    for t in (q, u):
        assert t.dim() == 2 and t.stride(1) == 1 and t.dtype == q.dtype and t.dtype in (torch.float32, torch.float16)
    for t in (kv0,) + ((kv1,) if kv1 is not None else ()):
        assert t.dim() == 2 and t.stride(1) == 1 and t.dtype == kv0.dtype and t.dtype in (torch.float32, torch.float16)
    if out is None:
        out = torch.empty(M, D + H * D, dtype=out_dtype, device=q.device)
    assert out.dtype in (torch.float32, torch.float16) and out.stride(1) == 1
    none_valid = torch.empty(M, dtype=torch.bool, device=q.device)
    assert idx.dtype == torch.int32 and idx.is_contiguous() and idx.shape[-1] == K0 + K1
    inv = _u8(invalid)
    assert inv.is_contiguous()
    if rel is not None:
        assert rel.is_contiguous() and rel.dtype == torch.float32
    if emb is not None:
        assert emb.is_contiguous() and emb.dtype == torch.float32
    z = out[:, D:]
    L.check(L.load().tb_knarpe_attn(
        L.ptr(q), q.stride(0), L.ptr(u), u.stride(0), L.ptr(kv0), kv0.stride(0), T0, div0, K0,
        L.ptr(kv1), kv1.stride(0) if kv1 is not None else 0, T1, div1, K1, L.ptr(idx), L.ptr(inv), L.ptr(rel),
        L.ptr(emb), L.ptr(freq_xy), B, S, D, H, L.ptr(out), L.ptr(z), out.stride(0), L.ptr(_u8(none_valid)),
        int(fast_trig) | (2 if rpe_mma else 0) | (4 if out.dtype == torch.float16 else 0) |
        (8 if q.dtype == torch.float16 else 0) | (16 if interleaved else 0), L.stream()), "tb_knarpe_attn")
    _count()
    return out, none_valid


def linear(x: Tensor, w: Tensor, b: Optional[Tensor] = None, relu: bool = False, mask_pre: Optional[Tensor] = None,
           res: Optional[Tensor] = None, mask_post: Optional[Tensor] = None, out: Optional[Tensor] = None,
           precision: int = 0, bias_group: int = 0, out_h: Optional[Tensor] = None, col_h: int = 0) -> Tensor:
    """Y = epilogue(X W^T + b) on 2-D row-strided views (see tb_linear). With `out_h` (float16 [M, N - col_h]) the
    columns >= col_h go there instead (tensor-core mode only) and `out` holds the first col_h columns
    (returned; None when col_h == 0). Inputs that require grad route to the differentiable form (autograd.linear)."""
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (x, w, b, res)):
        from . import autograd as AG
        assert out_h is None, "the training path keeps fp32 activations"
        return AG.linear(x, w, b, relu, mask_pre, res, mask_post, out, precision, bias_group)
    if precision == 3:  # fp32-accurate on the tf32 tensor cores (3xTF32); small / odd shapes stay on the FFMA kernel
        M_, K_ = x.shape
        if out_h is not None or K_ % 4 or x.stride(0) % 4 or M_ < 1024 or x.data_ptr() % 16:
            precision = 0
        else:
            return linear(tf32_split3(x), _w3(w), b, relu, mask_pre, res, mask_post, out, 1, bias_group)
    in_dt = torch.float16 if precision == 2 else torch.float32  # precision 2: fp16 activations x fp16 weights
    assert x.dim() == 2 and x.stride(1) == 1 and w.is_contiguous() and x.dtype == in_dt and w.dtype == in_dt, \
        (x.dtype, w.dtype, precision)
    M, K = x.shape
    N = w.shape[0]
    assert w.shape[1] == K, (w.shape, x.shape)
    n32 = N if out_h is None else col_h
    if out is None and n32 > 0:
        out = torch.empty(M, n32, dtype=torch.float32, device=x.device)
    assert out is None or (out.stride(1) == 1 and out.shape[0] == M and out.shape[1] == n32)
    if out_h is not None:
        assert out_h.dtype == torch.float16 and out_h.stride(1) == 1 and out_h.shape == (M, N - col_h)
    if res is not None:
        assert res.stride(1) == 1 and res.shape == (M, N)
    if bias_group:
        assert b is not None and b.is_contiguous() and b.shape == ((M + bias_group - 1) // bias_group, N), b.shape
    L.check(L.load().tb_linear(L.ptr(x), x.stride(0), L.ptr(w), L.ptr(b), bias_group, L.ptr(out),
                               out.stride(0) if out is not None else 0, M, N, K,
                               int(relu), L.ptr(_u8(mask_pre)), L.ptr(res), res.stride(0) if res is not None else 0,
                               L.ptr(_u8(mask_post)), precision, L.ptr(out_h),
                               out_h.stride(0) if out_h is not None else 0, col_h, L.stream()), "tb_linear")
    _count()
    return out


def tf32_split3(x: Tensor) -> Tensor:
    """[x | x - trunc_tf32(x) | x] rows (tb_tf32_split3): the activation operand of a 3xTF32 projection."""
    M, K = x.shape
    out = torch.empty(M, 3 * K, dtype=torch.float32, device=x.device)
    L.check(L.load().tb_tf32_split3(L.ptr(x), x.stride(0), M, K, L.ptr(out), 3 * K, L.stream()), "tb_tf32_split3")
    _count()
    return out


def _w3(w: Tensor) -> Tensor:
    """[W | W | W - trunc_tf32(W)] for a 3xTF32 projection, cached on the weight object until it is modified."""
    c = getattr(w, "_tb_w3", None)
    if c is None or c[0] != w._version:
        hi = (w.detach().view(torch.int32) & -8192).view(torch.float32)  # keep sign, exponent and 10 mantissa bits
        c = (w._version, torch.cat([w.detach(), w.detach(), w.detach() - hi], 1).contiguous())
        w._tb_w3 = c
    return c[1]


def linear_ln(x: Tensor, w: Tensor, b: Optional[Tensor], gamma: Tensor, beta: Tensor, mask_pre: Optional[Tensor] = None,
              res: Optional[Tensor] = None, mask_post: Optional[Tensor] = None, out: Optional[Tensor] = None,
              precision: int = 2) -> Tuple[Tensor, Tensor]:
    """tb_linear_ln: (Y, fp16 LayerNorm(Y) * gamma + beta) from one launch; N must be 128 (tensor-core mode)."""
    in_dt = torch.float16 if precision == 2 else torch.float32
    assert x.dim() == 2 and x.stride(1) == 1 and w.is_contiguous() and x.dtype == in_dt and w.dtype == in_dt
    M, K = x.shape
    N = w.shape[0]
    assert w.shape[1] == K and gamma.shape == (N,) and beta.shape == (N,)
    if out is None:
        out = torch.empty(M, N, dtype=torch.float32, device=x.device)
    assert out.stride(1) == 1 and out.shape == (M, N)
    if res is not None:
        assert res.stride(1) == 1 and res.shape == (M, N)
    ln_out = torch.empty(M, N, dtype=torch.float16, device=x.device)
    L.check(L.load().tb_linear_ln(L.ptr(x), x.stride(0), L.ptr(w), L.ptr(b), L.ptr(out), out.stride(0), M, N, K,
                                  L.ptr(_u8(mask_pre)), L.ptr(res), res.stride(0) if res is not None else 0,
                                  L.ptr(_u8(mask_post)), precision, L.ptr(_f32c(gamma)), L.ptr(_f32c(beta)),
                                  L.ptr(ln_out), ln_out.stride(0), L.stream()), "tb_linear_ln")
    _count()
    return out, ln_out


def layernorm(x: Tensor, gamma: Tensor, beta: Tensor, out: Optional[Tensor] = None, relu: bool = False,
              out_dtype: torch.dtype = torch.float32) -> Tensor:
    if torch.is_grad_enabled() and (x.requires_grad or gamma.requires_grad or beta.requires_grad):
        from . import autograd as AG
        assert out_dtype == torch.float32, "the training path keeps fp32 activations"
        return AG.layernorm(x, gamma, beta, relu, out)
    assert x.dim() == 2 and x.stride(1) == 1 and x.dtype == torch.float32
    M, D = x.shape
    if out is None:
        out = torch.empty(M, D, dtype=out_dtype, device=x.device)
    assert out.dtype in (torch.float32, torch.float16) and out.stride(1) == 1
    L.check(L.load().tb_layernorm(L.ptr(x), x.stride(0), L.ptr(gamma), L.ptr(beta), L.ptr(out), out.stride(0), M, D,
                                  int(relu) | (2 if out.dtype == torch.float16 else 0), L.stream()), "tb_layernorm")
    _count()
    return out


def pointnet_pool(x: Tensor, invalid: Tensor, G: int, Lg: int, mode: int) -> Optional[Tensor]:
    """x [G*L, C2] modified in place (mode 0) / max-pooled over valid rows to [G, C2] (mode 1) or [G, 2*C2] = [m|m]
    (mode 2)."""
    if torch.is_grad_enabled() and x.requires_grad:
        from . import autograd as AG
        return AG.pointnet_pool(x, invalid, G, Lg, mode)
    assert x.dim() == 2 and x.stride(1) == 1 and x.shape[0] == G * Lg
    C2 = x.shape[1]
    out = torch.empty(G, C2 * mode, dtype=torch.float32, device=x.device) if mode else None
    inv = _u8(invalid)
    assert inv.is_contiguous() and inv.numel() == G * Lg
    L.check(L.load().tb_pointnet_pool(L.ptr(x), x.stride(0), L.ptr(inv), G, Lg, C2, mode, L.ptr(out),
                                      out.stride(0) if out is not None else 0, L.stream()), "tb_pointnet_pool")
    _count()
    return out


def pose_emb(pose: Tensor, freq_xy: Tensor, pe_dim: int, frame: Optional[Tensor] = None, frame_div: int = 1,
             out: Optional[Tensor] = None) -> Tensor:
    pose = _f32c(pose).view(-1, 3)
    M = pose.shape[0]
    if out is None:
        out = torch.empty(M, pe_dim, dtype=torch.float32, device=pose.device)
    if frame is not None:
        frame = _f32c(frame).view(-1, 3)
    L.check(L.load().tb_pose_emb(L.ptr(pose), L.ptr(frame), frame_div, L.ptr(freq_xy), M, pe_dim, L.ptr(out),
                                 out.stride(0), L.stream()), "tb_pose_emb")
    _count()
    return out


def gather_rows(table: Tensor, idx: Tensor, rows_per_batch: int, div: int = 1, out: Optional[Tensor] = None) -> Tensor:
    """table [Bt, T, C] (contiguous), idx int32 [M] -> out [M, C]; batch of row m is (m // rows_per_batch) // div."""
    assert table.dim() == 3 and table.is_contiguous() and idx.dtype == torch.int32 and idx.is_contiguous()
    Bt, T, C = table.shape
    M = idx.numel()
    if out is None:
        out = torch.empty(M, C, dtype=torch.float32, device=table.device)
    L.check(L.load().tb_gather_rows(L.ptr(table), C, T, L.ptr(idx), M, rows_per_batch, div, C, L.ptr(out),
                                    out.stride(0), L.stream()), "tb_gather_rows")
    _count()
    return out


def copy_rows(items, src_rollout: Optional[Tensor] = None, R: int = 0) -> None:
    """tb_copy_rows: one launch for all `items` = [(src, dst, per_rollout)], contiguous tensors of equal shape and
    dtype whose rows run along dim 0. With `src_rollout` (int32 [rows], on the device) the per-rollout items gather
    row sc * R + src_rollout[b] into row b = sc * R + r; the others, and all of them without a map, are plain copies."""
    arr = (L.RowCopy * len(items))()
    for i, (src, dst, per_rollout) in enumerate(items):
        assert src.shape == dst.shape and src.dtype == dst.dtype and src.is_contiguous() and dst.is_contiguous()
        rows = src.shape[0]
        arr[i] = L.RowCopy(src.data_ptr(), dst.data_ptr(), src.numel() * src.element_size() // rows, rows,
                           int(per_rollout))
    if src_rollout is not None:
        assert src_rollout.dtype == torch.int32 and src_rollout.is_contiguous()
    L.check(L.load().tb_copy_rows(arr, len(items), L.ptr(src_rollout), R, L.stream()), "tb_copy_rows")
    _count()


def host_f3(vals):
    return (ctypes.c_float * 3)(*[float(v) for v in vals])


def future_filter(collided: Tensor, run_road_edge: Tensor, role_any: Tensor, n_sc: int, K: int, t0: int,
                  w_road_edge: float, n_keep: int) -> Tuple[Tensor, Tensor]:
    """tb_future_filter: flags [n_sc*K, A, T] (bool/u8), role_any [n_sc, A] -> (score [n_sc, K], sel int32 [n_sc, n_keep])."""
    col, edge, role = _u8(collided), _u8(run_road_edge), _u8(role_any)
    assert col.is_contiguous() and edge.is_contiguous() and role.is_contiguous() and col.shape == edge.shape
    B, A, T = col.shape
    assert B == n_sc * K and role.shape == (n_sc, A)
    score = torch.empty(n_sc, K, dtype=torch.float32, device=col.device)
    sel = torch.empty(n_sc, n_keep, dtype=torch.int32, device=col.device)
    L.check(L.load().tb_future_filter(L.ptr(col), L.ptr(edge), L.ptr(role), n_sc, K, A, T, t0, float(w_road_edge), n_keep,
                                      L.ptr(score), L.ptr(sel), L.stream()), "tb_future_filter")
    _count(2)
    return score, sel


def traj_global(pose: Tensor, sel: Optional[Tensor], center: Tensor, yaw: Tensor, n_sc: int, K: int, t0: int
                ) -> Tuple[Tensor, Tensor]:
    """tb_traj_global: pose [n_sc*K, A, T, 3] scene-centric -> (pos [n_sc, n_keep, A, T-t0, 2], yaw [.., 1]) global."""
    pose, center, yaw = _f32c(pose), _f32c(center), _f32c(yaw).reshape(-1)
    B, A, T, _ = pose.shape
    n_keep = K if sel is None else sel.shape[1]
    assert B == n_sc * K and (sel is None or (sel.dtype == torch.int32 and sel.is_contiguous()))
    pos = torch.empty(n_sc, n_keep, A, T - t0, 2, dtype=torch.float32, device=pose.device)
    oyaw = torch.empty(n_sc, n_keep, A, T - t0, 1, dtype=torch.float32, device=pose.device)
    L.check(L.load().tb_traj_global(L.ptr(pose), L.ptr(sel), L.ptr(center), L.ptr(yaw), n_sc, K, n_keep, A, T, t0,
                                    L.ptr(pos), L.ptr(oyaw), L.stream()), "tb_traj_global")
    _count()
    return pos, oyaw


def womd_post(trajs: Tensor, scores: Optional[Tensor], ag_type: Tensor, k_pred: int = 6, use_ade: bool = True,
              mpa_nms_thresh=(2.0, 2.0, 2.0), score_temperature: float = -1.0, t_first: int = 4, t_stride: int = 5,
              t_end: int = 80) -> Tuple[Tensor, Tensor, Tensor]:
    """tb_womd_post (womd_post_processing.py:36-106): trajs [n_sc, K, A, T, 3], scores [n_sc, K, A] log-probs or None,
    ag_type [n_sc, A, 3] -> (trajs [n_sc, A, k, n_out, 3], scores [n_sc, A, k], mode [n_sc, A, k] int32)."""
    trajs = _f32c(trajs)
    n_sc, K, A, T, _ = trajs.shape
    scores = None if scores is None else _f32c(scores)
    assert scores is None or scores.shape == (n_sc, K, A)
    ag_type = _u8(ag_type.contiguous())
    assert ag_type.shape == (n_sc, A, 3)
    k = min(K, k_pred)
    n_out = len(range(t_first, min(t_end, T), t_stride))
    out_t = torch.empty(n_sc, A, k, n_out, 3, dtype=torch.float32, device=trajs.device)
    out_s = torch.empty(n_sc, A, k, dtype=torch.float32, device=trajs.device)
    out_m = torch.empty(n_sc, A, k, dtype=torch.int32, device=trajs.device)
    thr = list(mpa_nms_thresh) + [0.0] * 3
    L.check(L.load().tb_womd_post(L.ptr(trajs), L.ptr(scores), L.ptr(ag_type), n_sc, K, A, T, k_pred, int(use_ade),
                                  int(len(mpa_nms_thresh) > 0), float(thr[0]), float(thr[1]), float(thr[2]),
                                  float(score_temperature), t_first, t_stride, t_end, L.ptr(out_t), L.ptr(out_s),
                                  L.ptr(out_m), L.stream()), "tb_womd_post")
    _count()
    return out_t, out_s, out_m


def knarpe_attn_bwd(q: Tensor, u: Tensor, kv0: Tensor, T0: int, div0: int, K0: int, idx: Tensor, invalid: Tensor,
                    rel: Tensor, freq_xy: Tensor, B: int, S: int, D: int, d_out: Tensor, H: int = 4,
                    kv1: Optional[Tensor] = None, T1: int = 0, div1: int = 1, K1: int = 0
                    ) -> Tuple[Tensor, Tensor, Optional[Tensor]]:
    """Backward of the KNARPE core (tb_knarpe_attn_bwd): d_out [B*S, D+H*D] = [d_ov | d_z] ->
    (d_qu [B*S, D+H*D] = [d_q | d_u], d_kv0 like kv0, d_kv1 like kv1 or None). fp32 tables only."""
    M = B * S
    for t in (q, u, kv0, d_out) + ((kv1,) if kv1 is not None else ()):
        assert t.dim() == 2 and t.stride(1) == 1 and t.dtype == torch.float32
    assert kv0.is_contiguous() and (kv1 is None or kv1.is_contiguous())
    d_qu = torch.empty(M, D + H * D, dtype=torch.float32, device=q.device)
    d_kv0 = torch.zeros_like(kv0)
    d_kv1 = torch.zeros_like(kv1) if kv1 is not None else None
    inv = _u8(invalid)
    assert idx.dtype == torch.int32 and idx.is_contiguous() and inv.is_contiguous() and rel.is_contiguous()
    L.check(L.load().tb_knarpe_attn_bwd(
        L.ptr(q), q.stride(0), L.ptr(u), u.stride(0), L.ptr(kv0), kv0.stride(0), T0, div0, K0,
        L.ptr(kv1), kv1.stride(0) if kv1 is not None else 0, T1, div1, K1, L.ptr(idx), L.ptr(inv), L.ptr(rel),
        L.ptr(freq_xy), B, S, D, H, L.ptr(d_out), L.ptr(d_out[:, D:]), d_out.stride(0), L.ptr(d_qu), d_qu.stride(0),
        L.ptr(d_kv0), L.ptr(d_kv1), L.stream()), "tb_knarpe_attn_bwd")
    _count()
    return d_qu, d_kv0, d_kv1


# ---------------------------------------------------------------------------------------------------- fused MLP chain
class _ChainUnit(ctypes.Structure):
    """tb_chain_unit of include/tb_knarpe.h."""
    _fields_ = [("kind", ctypes.c_int), ("W", ctypes.c_void_p), ("K", ctypes.c_int), ("N", ctypes.c_int),
                ("n0", ctypes.c_int), ("a_buf", ctypes.c_int * 4), ("bias", ctypes.c_void_p), ("relu", ctypes.c_int),
                ("n_valid", ctypes.c_int), ("mask_pre", ctypes.c_int), ("mask_post", ctypes.c_int), ("res", ctypes.c_int),
                ("ldr", ctypes.c_int), ("res_col", ctypes.c_int), ("out_buf", ctypes.c_int), ("out_g", ctypes.c_int),
                ("ldg", ctypes.c_int), ("g_col", ctypes.c_int), ("out_h", ctypes.c_int), ("ldh", ctypes.c_int),
                ("h_col", ctypes.c_int), ("ln_out", ctypes.c_int), ("ld_ln", ctypes.c_int), ("ln_gamma", ctypes.c_void_p),
                ("ln_beta", ctypes.c_void_p), ("src", ctypes.c_int), ("lds", ctypes.c_int), ("src_col", ctypes.c_int),
                ("src_f16", ctypes.c_int)]


class ChainProgram:
    """Builder / runner of a fused MLP chain (tb_chain_encode / tb_chain_run): `load` and `gemm` append units,
    `finish` encodes the program (TMA descriptors of the weights included) and uploads it, `run` launches it on a set of
    binding tensors. Weights are fp16 [N, K] row-major device tensors kept alive by the program.
    `spec` keeps every unit as a plain dict of the builder's arguments (weights, biases and LayerNorm parameters as the
    tensors given), so a reference can run the same program (tests/_chain_ref.py). A program that is only described
    (never finished) may hold weights of any float dtype on any device."""

    def __init__(self, device, n_buf: int = 4):
        self.dev, self.n_buf = torch.device(device), n_buf
        self.units, self.keep, self.spec = [], [], []
        self.blob = self.host = None

    def _unit(self, **kw) -> _ChainUnit:
        u = _ChainUnit()
        for f in ("mask_pre", "mask_post", "res", "out_buf", "out_g", "out_h", "ln_out", "src"):
            setattr(u, f, -1)
        for i in range(4):
            u.a_buf[i] = -1
        for k, v in kw.items():
            setattr(u, k, v)
        self.units.append(u)
        return u

    def load(self, src: int, lds: int, out_buf: int, src_col: int = 0, f16: bool = False) -> None:
        self._unit(kind=1, src=src, lds=lds, src_col=src_col, src_f16=int(f16), out_buf=out_buf)
        self.spec.append(dict(kind="load", src=src, lds=lds, out_buf=out_buf, src_col=src_col, f16=bool(f16)))

    def gemm(self, w: Tensor, a_bufs, bias: Optional[Tensor] = None, n0: int = 0, relu: bool = False, out_buf: int = -1,
             mask_pre: int = -1, mask_post: int = -1, res: int = -1, ldr: int = 0, res_col: int = 0, out_g: int = -1,
             ldg: int = 0, g_col: int = 0, n_valid: int = 0, out_h: int = -1, ldh: int = 0, h_col: int = 0, ln_out: int = -1,
             ld_ln: int = 0, ln_gamma: Optional[Tensor] = None, ln_beta: Optional[Tensor] = None) -> None:
        """w [N, K]: K columns from the buffers a_bufs side by side, 128 per buffer (the last one may contribute only
        its first 64 columns: K = 64, 192, 320, 448)."""
        assert w.is_contiguous() and w.dim() == 2
        N, K = w.shape
        assert len(a_bufs) == (K + 127) // 128, (w.shape, a_bufs)
        self.spec.append(dict(kind="gemm", w=w, a_bufs=list(a_bufs), bias=bias, n0=n0, relu=bool(relu), out_buf=out_buf,
                              mask_pre=mask_pre, mask_post=mask_post, res=res, ldr=ldr, res_col=res_col, out_g=out_g,
                              ldg=ldg, g_col=g_col, n_valid=n_valid, out_h=out_h, ldh=ldh, h_col=h_col, ln_out=ln_out,
                              ld_ln=ld_ln, ln_gamma=ln_gamma, ln_beta=ln_beta))
        u = self._unit(kind=0, W=w.data_ptr(), K=K, N=N, n0=n0, relu=int(relu), out_buf=out_buf, mask_pre=mask_pre,
                       mask_post=mask_post, res=res, ldr=ldr, res_col=res_col, out_g=out_g, ldg=ldg, g_col=g_col,
                       n_valid=n_valid, out_h=out_h, ldh=ldh, h_col=h_col, ln_out=ln_out, ld_ln=ld_ln)
        for i, b in enumerate(a_bufs):
            u.a_buf[i] = b
        self.keep.append(w)
        if bias is not None:  # the epilogue reads bias[n0 : n0 + 128] unconditionally
            b = bias.detach().to(self.dev, torch.float32).contiguous()
            if b.numel() < n0 + 128:
                b = torch.cat([b, b.new_zeros(n0 + 128 - b.numel())])
            self.keep.append(b)
            u.bias = b.data_ptr()
        if ln_out >= 0:
            g, be = (t.detach().to(self.dev, torch.float32).contiguous() for t in (ln_gamma, ln_beta))
            self.keep += [g, be]
            u.ln_gamma, u.ln_beta = g.data_ptr(), be.data_ptr()

    def finish(self) -> "ChainProgram":
        for s in self.spec:
            assert s["kind"] == "load" or (s["w"].dtype == torch.float16 and s["w"].is_cuda), \
                "a program that runs needs fp16 device weights"
        lib = L.load()
        n = lib.tb_chain_program_bytes()
        self.host = (ctypes.c_uint8 * n)()
        arr = (_ChainUnit * len(self.units))(*self.units)
        L.check(lib.tb_chain_encode(arr, len(self.units), self.n_buf, self.host), "tb_chain_encode")
        self.blob = torch.frombuffer(bytearray(self.host), dtype=torch.uint8).to(self.dev)
        assert self.blob.data_ptr() % 128 == 0
        return self

    def run(self, bindings, M: int) -> None:
        ptrs = (ctypes.c_void_p * len(bindings))(*[None if t is None else t.data_ptr() for t in bindings])
        L.check(L.load().tb_chain_run(L.ptr(self.blob), self.host, ptrs, len(bindings), M, L.stream()), "tb_chain_run")
        _count()
