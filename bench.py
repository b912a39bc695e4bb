#!/usr/bin/env python
"""Benchmark of the closed-loop WOSAC rollout hot path (BASELINE.json metric: scenario-rollout-steps/s).

  python bench.py --gpus N --steps K --warmup W            # our CUDA path (N>1: launched by torchrun, one rank/GPU)
  python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPU cores (oracle port)
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/*.npy

A bench "step" = ONE complete closed-loop rollout of the per-GPU workload (BASELINE config 3: 16 scenes x 32 rollouts,
128 agents, 1024 polylines x 20 nodes, 40 traffic lights, 11-step history): 90 policy iterations of which the 80
post-history ones count. value = scenes x 32 x 80 / time, summed over ranks (weak scaling: 16 scenes per GPU).
  value : rollout loop only, scene tokens and inputs resident in HBM (what `WaymoMotion.rollout` times)
  e2e   : RolloutEngine.rollout(host batch): H2D of the pinned inputs + map/TL scene encoding + 90 steps + D2H of the
          80-step trajectories, every step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import tbpkg  # noqa: E402,F401
from trafficbotsv1_5_b200 import config, params, synth  # noqa: E402

METRIC = "closed_loop_scenario_rollout_steps_per_sec"
UNIT = "rollout-scene-steps/s"
N_COUNTED, N_ITER = 80, 90


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scenes", type=int, default=16, help="scenes per GPU")
    ap.add_argument("--rollouts", type=int, default=32)
    ap.add_argument("--precision", type=int, default=1,
                    help="1 (default): tcgen05 kind::tf32 / kind::f16 projections with fp16 K|V, q|u, ov|z, FFN-hidden and "
                         "LayerNorm rows (fp32 accumulators, residual stream and rollout state); 0: fp32 everywhere")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the fp32 / rule-check extra measurements")
    ap.add_argument("--scenes-total", type=int, default=0,
                    help="BASELINE config 5: sweep this many scenes (512) sharded over the ranks in batches of --scenes, "
                         "NCCL gather of every batch's trajectories overlapped with the next batch (strong scaling)")
    ap.add_argument("--train", action="store_true",
                    help="BASELINE config 4 instead of the rollout: forward + backward of the training_step body "
                         "(--scenes scenes per GPU, default 64; dropout 0) - prints its own JSON line")
    ap.add_argument("--rule-checks", action="store_true",
                    help="also run the logging-only TrafficRuleChecker checks (collision, road edge, ...) every step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32, or "
                         "float64 where the output is), at most 64 MB in all: larger outputs are cut to a fixed, seeded "
                         "sample of rows. Inputs depend only on the arguments, so two builds can be compared file by file")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA path, not to --impl reference")
    return args


DUMP_BYTES = 64 * 10**6  # 64 MB, npy headers included


def dump_outputs(out_dir, whole, rows=None, seed=0):
    """Write every tensor of `whole` and `rows` to out_dir/<name>.npy: float64 stays float64, everything else (fp32,
    fp16, bool, int) becomes float32. The tensors of `rows` share their leading dimension; if the files would exceed
    DUMP_BYTES in all, those tensors are cut to the same rows, drawn by a generator seeded with `seed` and kept in
    ascending order, so the sample depends only on the shapes. Returns a short description for the log."""
    import numpy as np
    rows = rows or {}

    def host(t):
        return t.detach().to("cpu", torch.float64 if t.dtype == torch.float64 else torch.float32)

    whole = {k: host(v) for k, v in whole.items()}
    nbytes = lambda ts: sum(t.numel() * t.element_size() for t in ts)  # noqa: E731
    budget = DUMP_BYTES - nbytes(whole.values()) - 256 * (len(whole) + len(rows))  # npy headers
    n = next(iter(rows.values())).shape[0] if rows else 0
    per_row = sum(v[0].numel() * (8 if v.dtype == torch.float64 else 4) for v in rows.values())
    keep = min(n, budget // per_row) if rows else 0
    if rows and keep < 1:
        raise ValueError(f"--dump-outputs: the outputs do not fit {DUMP_BYTES / 1e6:.0f} MB even at one row")
    sel = None
    if keep < n:
        sel = torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:keep].sort().values
    out = dict(whole, **{k: host(v if sel is None else v[sel.to(v.device)]) for k, v in rows.items()})
    os.makedirs(out_dir, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), v.numpy())
    what = f"{len(out)} arrays, {nbytes(out.values()) / 1e6:.1f} MB"
    return what if sel is None else what + f"; {keep} of {n} rows of {', '.join(rows)} (seed {seed})"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self._stop = index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self.t.join(timeout=6)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(sm))


# ------------------------------------------------------------------------------------------------------ CPU arm
def cpu_rollout_rate(n_threads, n_sc=1, R=8, iters=6, rule_checks=False):
    """The reference algorithm (oracle port, torch CPU fp32) on a bounded sample of the same workload shape:
    n_sc scene x R rollouts x `iters` policy iterations (history warm-up included, scene encoding excluded, like
    `value`). Rate is scaled to the metric's 80-of-90 accounting."""
    from oracle import tb_oracle as O
    torch.set_num_threads(n_threads)
    cfg = config.default_model_cfg()
    sz = config.derived_sizes(cfg)
    P = params.init_params(cfg, 0)
    batch = synth.make_scene_batch(n_sc=n_sc, seed=1000)
    with torch.no_grad():
        mp = O.map_encoder(P, cfg, sz, batch["sc/mp_valid"], batch["sc/mp_attr"], batch["sc/mp_pose"])
        tl = O.tl_pre_compute(P, cfg, sz, batch["sc/tl_valid"], batch["sc/tl_attr"], batch["sc/tl_pose"], mp)
        mp = {k: mp[k] for k in ("mp_token_invalid", "mp_token_feature", "mp_token_pose")}
        O.rollout(P, cfg, sz, config.DYNAMICS_CFG, config.ROLLOUT_CFG, batch, R, 1, mp=mp, tl=tl, rule_checks=rule_checks)  # warm-up
        t0 = time.perf_counter()
        O.rollout(P, cfg, sz, config.DYNAMICS_CFG, config.ROLLOUT_CFG, batch, R, iters, mp=mp, tl=tl, rule_checks=rule_checks)
        dt = time.perf_counter() - t0
    per_iter = dt / iters
    rate = n_sc * R * N_COUNTED / (N_ITER * per_iter)
    sample = (f"{n_sc} scene x {R} rollouts x {iters} policy iterations (128 agents, 1024 polylines, 40 TL) in "
              f"{dt:.1f} s; scaled to 80 counted of 90 iterations")
    return rate, sample, per_iter


def eager_cuda_rate(dev, n_sc, R, iters, autocast):
    """The bar SURVEY 8(d) / BASELINE.md 3.2 name: the reference's own operation order (gather-then-project KNARPE,
    materialised [B,S,T,3] relative poses + topk, per-step re-encoding; the oracle port of it) as eager PyTorch on the
    SAME B200 — fp32, or fp16 autocast as the reference trains (configs/trainer/default.yaml:16). Same accounting
    as `value`: scene tokens resident, `iters` policy iterations timed with CUDA events, scaled to 80-of-90. Falls back
    to fewer scenes if the reference-order activations do not fit."""
    from oracle import tb_oracle as O
    cfg = config.default_model_cfg()
    sz = config.derived_sizes(cfg)
    P = {k: v.to(dev) for k, v in params.init_params(cfg, 0).items()}
    host_batch = synth.make_scene_batch(n_sc=n_sc, seed=1000, n_rollout=R)
    prev = torch.get_default_device()
    torch.set_default_device(dev)  # the oracle's factory calls (eye, arange, zeros) then allocate on the GPU
    try:
        while n_sc >= 1:
            try:
                batch = {k: v[:n_sc].to(dev) for k, v in host_batch.items()}
                with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
                    mp = O.map_encoder(P, cfg, sz, batch["sc/mp_valid"], batch["sc/mp_attr"], batch["sc/mp_pose"])
                    tl = O.tl_pre_compute(P, cfg, sz, batch["sc/tl_valid"], batch["sc/tl_attr"], batch["sc/tl_pose"], mp)
                    mp = {k: mp[k] for k in ("mp_token_invalid", "mp_token_feature", "mp_token_pose")}
                    run = lambda n: O.rollout(P, cfg, sz, config.DYNAMICS_CFG, config.ROLLOUT_CFG, batch, R, n, mp=mp, tl=tl)  # noqa: E731
                    run(2)  # warm-up (cuBLAS handles, allocator)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize()
                    e0.record()
                    run(iters)
                    e1.record()
                    torch.cuda.synchronize()
                per_iter = e0.elapsed_time(e1) * 1e-3 / iters
                peak_gb = torch.cuda.max_memory_allocated(dev) / 2**30
                return dict(value=n_sc * R * N_COUNTED / (N_ITER * per_iter), unit=UNIT, ms_per_policy_iteration=per_iter * 1e3,
                            scenes=n_sc, rollouts=R, policy_iterations_timed=iters, peak_mem_gib=round(peak_gb, 1),
                            what="reference operation order (oracle port) as eager PyTorch on this GPU, "
                                 + ("fp16 autocast" if autocast else "fp32") + "; scaled to 80 counted of 90 iterations")
            except torch.OutOfMemoryError:
                torch.cuda.empty_cache()
                n_sc //= 2
        return dict(unavailable="out of memory at 1 scene")
    finally:
        torch.set_default_device(prev)
        torch.cuda.empty_cache()


def knarpe_microbench(dev, peaks):
    """BASELINE config 2: KNARPE attention, 2048 tokens, K = 36 neighbours, 4 heads, d = 256, fp32 and 16-bit (IEEE
    fp16: same bytes as bf16, 3 more mantissa bits) on one B200. (i) whole `AttentionRPE.forward` of the drop-in module
    with the reference's pre-gathered [B,S,K,d] target (projections included), (ii) the attention core alone on a
    2048-row K|V table (post-projection), against SURVEY 8(d)'s algorithmic bytes: 156.4 MB fp32 / 78.8 MB 16-bit =
    23.9 / 12.1 us at the HBM peak. The unique bytes (~10 MB) are L2-resident, so "warm" (back-to-back launches) and
    "cold" (a 256 MB write between launches evicts L2) are both reported."""
    from trafficbotsv1_5_b200 import ops, reference_api as R
    d, H, S, K = 256, 4, 2048, 36
    g = torch.Generator().manual_seed(2)
    att = R.AttentionRPE(d, H, dropout_p=0.1, bias=True, d_rpe=d).eval()
    att.load_state_dict(params.rand_like_state_dict({k: tuple(v.shape) for k, v in att.state_dict().items()}, seed=11))
    att = att.to(dev)
    src = torch.randn(1, S, d, generator=g).to(dev)
    table = torch.randn(S, d, generator=g).to(dev)
    idx = torch.stack([torch.randperm(S, generator=g)[:K] for _ in range(S)]).to(dev)            # distinct neighbours
    mask = (torch.rand(1, S, K, generator=g) < 0.1).to(dev)
    rel = torch.cat([(torch.rand(1, S, K, 2, generator=g) * 2 - 1) * 100, (torch.rand(1, S, K, 1, generator=g) * 2 - 1) * 3.1],
                    -1).to(dev)
    tgt = table[idx].view(1, S, K, d).contiguous()
    flush = torch.empty(64 * 2**20, device=dev)  # 256 MB > the 126 MB L2
    peak = peaks.get("hbm_gbs", 6650.0)

    def time_us(fn, cold):
        """median-free device time of one call: `cold` brackets every launch with events after an L2-evicting fill;
        warm = 20 launches enqueued behind one long fill (so the CPU launch path is hidden) / 20."""
        for _ in range(3):
            fn()
        if cold:
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(20)]
            torch.cuda.synchronize()
            for a, b in ev:
                flush.fill_(1.0)
                a.record()
                fn()
                b.record()
            torch.cuda.synchronize()
            ts = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
            return ts[len(ts) // 2]
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        for _ in range(4):
            flush.fill_(1.0)  # ~0.3 ms of GPU work: the 20 launches below are queued before it drains
        fn()                  # re-warm L2 after the fills
        a.record()
        for _ in range(20):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e3 / 20

    out = {}
    freq = ops.pe_freq_xy(d, 1e3, dev)
    idx32 = idx.to(torch.int32).view(1, S, K).contiguous()
    for name, prec, esz in (("fp32", 0, 4), ("16bit", 1, 2)):
        att.precision, att._tb_ver = prec, None
        m = att._runner(d)
        f = m.fa[""]
        whole = lambda: att(src, tgt, tgt_padding_mask=mask, rpe=rel)  # noqa: E731
        # core only: [q|u] rows and the 2048-row K|V table as the projections of this mode produce them
        if prec:
            qu = torch.empty(S, d + H * d, dtype=torch.float16, device=dev)
            ops.linear(src.view(S, d), f["w_in_q"], f["b_in_q"], precision=1, out_h=qu, col_h=0)
            kv = torch.empty(S, 2 * d, dtype=torch.float16, device=dev)
            ops.linear(table, f["w_kv"], f["b_kv"], precision=1, out_h=kv, col_h=0)
        else:
            qu = ops.linear(src.view(S, d), f["w_in_q"], f["b_in_q"])
            kv = ops.linear(table, f["w_kv"], f["b_kv"])
        o = torch.empty(S, d + H * d, dtype=qu.dtype, device=dev)
        core = lambda: ops.knarpe_attn(qu[:, :d], qu[:, d:], kv, S, 1, K, idx32, mask, rel, freq, 1, S, d, H, out=o,  # noqa: E731
                                       fast_trig=bool(prec))
        alg = S * K * 2 * d * esz + S * 2 * d * esz + S * K * 5 + S * K * 12  # SURVEY 8(d)
        r = dict(algorithmic_bytes=alg, bound_us=alg / (peak * 1e3))
        for what, fn in (("whole_forward", whole), ("core", core)):
            for cold in (False, True):
                r[f"{what}_us_{'cold' if cold else 'warm'}"] = round(time_us(fn, cold), 2)
        r["core_as_issued_gbs_warm"] = round(alg / r["core_us_warm"] / 1e3, 1)
        r["core_frac_of_hbm_peak_warm"] = round(alg / r["core_us_warm"] / 1e3 / peak, 3)
        r["core_frac_of_hbm_peak_cold"] = round(alg / r["core_us_cold"] / 1e3 / peak, 3)
        out[name] = r
    out["config"] = dict(tokens=S, K=K, heads=H, d_model=d, masked=0.1, sixteen_bit="IEEE fp16 tables / rows, fp32 accumulate",
                         whole_forward="drop-in AttentionRPE.forward on the pre-gathered [1,2048,36,256] target "
                                       "(gather-then-project, as the reference's API dictates)", peak_gbs=peak)
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    vals, sample, per_iter = [], "", 0.0
    for i in range(args.warmup + args.steps):
        rate, sample, per_iter = cpu_rollout_rate(cores, 1, 16, 12)
        if i >= args.warmup:
            vals.append(rate)
    v = sum(vals) / len(vals)
    line = dict(metric=METRIC, value=v, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=per_iter * 1e3 * 12, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload="closed-loop WOSAC rollout, 128 agents / 1024 polylines x 20 / 40 TL / 11-step "
                                     "history; CPU sample per step: " + sample),
                cpu_baseline=dict(value=v, unit=UNIT, cores=cores, kind="port", sample=sample),
                e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line), file=_OUT, flush=True)


# ------------------------------------------------------------------------------------------------------ GPU arm
def attention_roofline(eng, peaks):
    """Dominant kernel = KNARPE attention core on the agent cross-attention (K = 64 map + 25 TL neighbours).
    achieved = algorithmic bytes of one launch / CUDA-event time of that launch (same tensors as the step)."""
    from trafficbotsv1_5_b200 import ops
    m, st, static = eng.model, eng._st, eng._static
    aux = {}
    eng._reset(st)
    for _ in range(12):  # advance past the warm-start so histories are full
        knn_prev = st["knn_state"].clone()  # per-row select state as the step finds it (previous step's x, y, kth)
        eng._step(st, static, eng._navi, aux)
    d, B, A = m.d, st["B"], st["A"]
    M = B * A
    p = "ag_encoder.tf_ag2agmptl.layers.0"
    f = m.fa[f"{p}.attn"]
    x = aux["ag_feat"]
    proj = m._in_q(f, m.ln(x, f"{p}.norm1", half=m.kv_half), f"{p}.attn")  # [q|u] rows as the step produces them
    kv_tl = m.kv_table(aux["tl_feat"], p, "norm_tgt")
    sz = eng.sz
    n_mp, n_tl = static["mp"]["mp_token_pose"].shape[1], static["tl"]["n_tl"]
    out = torch.empty(M, 5 * d, device=x.device, dtype=torch.float16 if m.kv_half else torch.float32)

    def launch():
        ops.knarpe_attn(proj[:, :d], proj[:, d:], static["kv_mp"][0], n_mp, eng.R, sz["k_ag2mp"], aux["cidx"],
                        aux["cinv"], aux["crel"], m.freq_rpe, B, A, d, 4, kv1=kv_tl, T1=n_tl, div1=eng.R,
                        K1=sz["k_ag2tl"], out=out, fast_trig=m.precision == 1, interleaved=m.kv_il)
    for _ in range(3):
        launch()
    n = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        launch()
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / n * 1e-3
    K = sz["k_ag2mp"] + sz["k_ag2tl"]
    n_valid = int((~aux["cinv"]).sum())
    # algorithmic bytes (SURVEY.md 8(d)): K,V rows of the unmasked neighbours as issued + q,u in + ov,z out + idx/mask/rel
    kv_sz = static["kv_mp"][0].element_size()  # 2 in the tensor-core mode (fp16 K|V tables), 4 in the fp32 mode
    io_sz = proj.element_size() + out.element_size()  # q,u rows in + ov,z rows out (fp16 in the tensor-core mode)
    bytes_alg = n_valid * 2 * d * kv_sz + M * (d + 4 * d) * io_sz + M * K * (4 + 1 + 12)
    peak = peaks.get("hbm_gbs", 6650.0)
    ach = bytes_alg / t / 1e9
    traffic = None  # dram__bytes_read.sum + dram__bytes_write.sum of this launch from the committed ncu --set full capture
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))["knarpe_attn_ag_cross_bytes"]
    except Exception:
        pass
    kname = ("knarpe_attn_mma_pair_kernel" if proj.element_size() == 2 else "knarpe_attn_mma_kernel") if kv_sz == 2 \
        else "knarpe_attn_kernel<128,false>"
    # ---- the select kernel the north star names: agent -> map launch of a rollout step (T = 1024 targets, K = 64),
    # temporal-coherence path with the per-row state of the previous step restored before every launch
    mp = static["mp"]
    T_mp, K_mp = mp["mp_token_pose"].shape[1], sz["k_ag2mp"]
    o_idx = torch.empty(B, A, K_mp, dtype=torch.int32, device=x.device)
    o_inv = torch.empty(B, A, K_mp, dtype=torch.bool, device=x.device)
    o_rel = torch.empty(B, A, K_mp, 3, device=x.device)
    states = [knn_prev.clone() for _ in range(n + 3)]

    def select(i):
        ops.knn_select(aux["tok_pose"], aux["tok_inv"], mp["mp_sorted_pose"], mp["mp_sorted_invalid"], K_mp, sz["dl_ag"],
                       tgt_div=eng.R, out=(o_idx, o_inv, o_rel), index_map=mp["mp_sorted_index"], row_state=states[i],
                       sorted_by_x=True)
    for i in range(3):
        select(n + i)
    torch.cuda.synchronize()
    e0.record()
    for i in range(n):
        select(i)
    e1.record()
    torch.cuda.synchronize()
    t_sel = e0.elapsed_time(e1) / n * 1e-3
    n_src = int((~aux["tok_inv"]).sum())
    sel_bytes = M * (T_mp * 13 + K_mp * 17)  # SURVEY 8(d): targets as issued (x, y, yaw, invalid) + idx / mask / rel out
    try:
        _tr = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))
        sel_traffic, lin_traffic = _tr.get("knn_select_ag_map_bytes"), _tr.get("linear_in_self_bytes")
    except Exception:
        sel_traffic = lin_traffic = None
    # ---- the projection that writes most: self in-projection of an agent layer, fp16 rows in / out in the 16-bit mode
    roof_proj = None
    if m.kv_half:
        fs = m.fa[f"{p}.attn_src"]
        x0 = m.ln(x, f"{p}.norm_src", half=True)
        row = torch.empty(M, fs["w_in_self"].shape[0], dtype=torch.float16, device=x.device)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=x.device)

        def cold(fn, reps=7):  # L2 flushed before every launch: a projection inside the step starts from HBM too
            fn()
            ts = []
            for _ in range(reps):
                flush.zero_()
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1) * 1e-3)
            return sorted(ts)[len(ts) // 2]

        nq = d + 4 * d
        t_p = cold(lambda: m._proj(x0, f"{p}.attn_src.w_in_self", fs["w_in_self"], fs["b_in_self"], out_h=row, col_h=0,
                                   il_blocks=(0, nq, nq + d)))
        t_fill = cold(lambda: row.zero_())  # what HBM gives a kernel that only WRITES these bytes
        pb = x0.numel() * 2 + fs["w_in_self"].numel() * 2 + row.numel() * 2
        roof_proj = dict(bound="hbm", kernel=f"linear_tc_kernel<F16> (self in-projection, M={M}, N={row.shape[1]}, K={d}, fp16 rows)",
                         achieved=pb / t_p / 1e9, peak=peak, unit="GB/s", frac=pb / t_p / 1e9 / peak, traffic=lin_traffic,
                         us_per_launch=t_p * 1e6, algorithmic_bytes=pb, bytes_written=row.numel() * 2,
                         write_only_floor_us=t_fill * 1e6, frac_of_write_floor=t_fill / t_p,
                         note="write-dominated: `write_only_floor_us` is a fill of the output alone, measured here; the "
                              "copy peak is not reachable by a kernel that mostly writes (profiles/r2_notes.md 9)")
    roof_sel = dict(bound="hbm", kernel="knn_select_kernel<32> (agent -> map, T=1024, K=64, temporal-coherence path)",
                    achieved=sel_bytes / t_sel / 1e9, peak=peak, unit="GB/s", frac=sel_bytes / t_sel / 1e9 / peak,
                    traffic=sel_traffic, us_per_launch=t_sel * 1e6, algorithmic_bytes=sel_bytes, rows=M, valid_rows=n_src,
                    pairs_per_s=M * T_mp / t_sel,
                    note="as-issued target bytes are shared-memory / L2 traffic (the 13 KB target block of a scene is staged "
                         "once per 64 rows); the kernel is bound by compare / select instruction issue (DESIGN.md 5)")
    return roof_sel, roof_proj, dict(bound="hbm", kernel=f"{kname} (agent cross-attn, K=89, {8 * kv_sz}-bit K|V / q|u / ov|z rows)", achieved=ach, peak=peak,
                unit="GB/s", frac=ach / peak, traffic=traffic, us_per_launch=t * 1e6,
                note="as-issued gather bytes are served by L2 (~85 % hit): DRAM traffic is a fraction of them; the "
                     "kernel's real ceiling is instruction issue / latency, not HBM (DESIGN.md 5)", algorithmic_bytes=bytes_alg,
                valid_pairs=n_valid, pairs=M * K, peak_source="MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback")


def run_sweep(args):
    """BASELINE config 5 as written: `--scenes-total` scenes x 32 rollouts x 80 steps, scenes sharded over the ranks in
    contiguous blocks (parallel.shard_range), every rank walks its shard in batches of `--scenes`; the trajectories of
    batch i are all-gathered over NCCL on a side stream while batch i+1 computes (parallel.OverlappedGather; reference:
    torchmetrics cat states, waymo_motion.py:894-909, submission.py:45-46,169-170). A bench step = one whole sweep.
      value: batches resident in HBM; scene encoding of every batch, its 90 policy iterations and the gather are timed
      e2e  : batches start in pinned host memory (H2D per batch) and every rank's trajectories go back to the host."""
    import torch.distributed as dist
    from trafficbotsv1_5_b200 import ops, parallel
    from trafficbotsv1_5_b200.engine import RolloutEngine
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: there is no CPU fallback for the product path"
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    total, per_batch, R = args.scenes_total, args.scenes, args.rollouts
    lo, hi = parallel.shard_range(total, world, rank)
    assert total % (world * per_batch) == 0, "scenes-total must be a multiple of gpus x scenes-per-batch"
    n_batches = (hi - lo) // per_batch
    cfg = config.default_model_cfg()
    P = params.init_params(cfg, 0)
    eng = RolloutEngine(P, cfg, dev, precision=args.precision, n_rollout=R, step_end=N_ITER)
    host = [{k: v.pin_memory() for k, v in synth.make_scene_batch(n_sc=per_batch, seed=1000 + lo + b * per_batch,
                                                                    n_rollout=R).items()} for b in range(n_batches)]
    resident = [{k: v.to(dev) for k, v in hb.items()} for hb in host]
    A = host[0]["sc/ag_valid"].shape[1]
    og = parallel.OverlappedGather(n_batches, (per_batch * R, A, N_COUNTED, 3), torch.float32, dev)
    h2d = sum(v.numel() * v.element_size() for v in host[0].values()) * n_batches

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1) * 1e-3], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    def sweep(batches):
        for b in batches:
            res = eng.rollout(b)
            og.submit(res["pred_pose"][:, :, N_ITER - N_COUNTED:])
        return og.wait()

    # ---- verification sweep (untimed): the gathered store must hold every scene's bytes where the shard map says
    sums = []
    for b in resident:
        res = eng.rollout(b)
        out = res["pred_pose"][:, :, N_ITER - N_COUNTED:]
        sums.append(parallel.scene_checksums(out.reshape(per_batch, -1)))
        og.submit(out)
    store = og.wait()
    mine = torch.stack(sums)                                           # [n_batches, per_batch]
    all_sums = [torch.empty_like(mine) for _ in range(world)]
    if world > 1:
        dist.all_gather(all_sums, mine)
    else:
        all_sums = [mine]
    got = torch.stack([parallel.scene_checksums(store[:, r].reshape(n_batches * per_batch, -1)).view(n_batches, per_batch)
                       for r in range(world)])
    gather_ok = bool(torch.equal(got, torch.stack(all_sums)))
    distinct = int(torch.stack(all_sums).unique().numel())
    assert gather_ok, "gathered trajectories do not match the per-scene checksums of their source ranks"

    for _ in range(max(args.warmup - 1, 0)):
        sweep(resident)
    l0 = ops.LAUNCHES
    with ClockSampler(local) as cs:
        t_val = timed(lambda: sweep(resident), args.steps)
    launches = (ops.LAUNCHES - l0) + args.steps * n_batches * eng.graph_steps * eng.launches_per_step
    clocks = cs.summary()
    if args.dump_outputs and rank == 0:  # the last sweep's gathered trajectories, one row per (scene, rollout)
        print("dump-outputs:", dump_outputs(args.dump_outputs, {}, dict(pred_pose=og.store.flatten(0, 2))),
              file=sys.stderr, flush=True)
    units = total * R * N_COUNTED
    value = units * args.steps / t_val

    host_out = [torch.empty(per_batch * R, A, N_COUNTED, 3).pin_memory() for _ in range(2)]
    d2h_stream = torch.cuda.Stream(device=dev)

    def sweep_e2e():
        for i, b in enumerate(host):
            res = eng.rollout(b)  # pinned host batch: H2D inside
            og.submit(res["pred_pose"][:, :, N_ITER - N_COUNTED:])
            d2h_stream.wait_stream(og.side)
            with torch.cuda.stream(d2h_stream):  # this rank's trajectories back to the host, behind the gather
                host_out[i % 2].copy_(og.stage[i % 2], non_blocking=True)
            og.free[i % 2] = torch.cuda.Event()
            og.free[i % 2].record(d2h_stream)
        og.wait()
        torch.cuda.current_stream().wait_stream(d2h_stream)
        torch.cuda.current_stream().synchronize()

    sweep_e2e()
    t_e2e = timed(sweep_e2e, max(1, args.steps))
    e2e = dict(value=units * max(1, args.steps) / t_e2e, unit=UNIT, h2d_bytes_per_step=h2d,
               d2h_bytes_per_step=n_batches * host_out[0].numel() * 4)
    if rank == 0:
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=t_val / args.steps * 1e3, higher_is_better=True, scaling="strong", vs_baseline=None,
                    dtype="f32" if args.precision == 0 else "tf32+fp16", data="synthetic",
                    config=dict(workload=f"config 5: scenario-sharded rollout sweep, {total} scenes x {R} rollouts x 80 steps "
                                         f"(90 policy iterations), {per_batch} scenes per batch, {n_batches} batches per GPU, NCCL "
                                         f"all-gather of every batch's 80-step trajectories overlapped with the next batch",
                                scenes_total=total, scenes_per_batch=per_batch, batches_per_gpu=n_batches, rollouts=R,
                                policy_iterations=N_ITER, counted_steps=N_COUNTED,
                                gathered_bytes_per_gpu=int(store.numel() * 4), gather_verified=gather_ok,
                                distinct_scene_checksums=distinct,
                                l2="per-iteration working set (>1 GB of activations) exceeds the 126 MB L2; no flush",
                                launches_per_policy_iteration=eng.launches_per_step),
                    clocks=clocks, e2e=e2e, gpu_launches=launches)
        print(json.dumps(line), file=_OUT, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_ours(args):
    import torch.distributed as dist
    from trafficbotsv1_5_b200 import ops
    from trafficbotsv1_5_b200.engine import RolloutEngine
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: there is no CPU fallback for the product path"
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    cfg = config.default_model_cfg()
    P = params.init_params(cfg, 0)
    eng = RolloutEngine(P, cfg, dev, precision=args.precision, n_rollout=args.rollouts, step_end=N_ITER,
                        rule_checks=args.rule_checks)
    n_sc = args.scenes
    batch = synth.make_scene_batch(n_sc=n_sc, seed=1000 + rank * n_sc, n_rollout=args.rollouts)
    batch = {k: v.pin_memory() for k, v in batch.items()}
    h2d = sum(v.numel() * v.element_size() for v in batch.values())

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1) * 1e-3], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # ---- value: rollout loop only, inputs + scene tokens resident
    eng.prepare(batch)
    from trafficbotsv1_5_b200 import parallel
    A_ = batch["sc/ag_valid"].shape[1]
    og = parallel.OverlappedGather(1, (n_sc * args.rollouts, A_, N_COUNTED, 3), torch.float32, dev) if world > 1 else None

    def loop_step():
        res = eng.run()
        if world > 1:  # the only cross-GPU step: gather of the 80-step trajectories (waymo_motion.py:894-909)
            og.submit(res["pred_pose"][:, :, N_ITER - N_COUNTED:])
            og.wait()

    gather_ok = None
    if world > 1:  # once, untimed: the gathered bytes of every rank match the checksums that rank computed locally
        res = eng.run()
        mine = parallel.scene_checksums(res["pred_pose"][:, :, N_ITER - N_COUNTED:].reshape(n_sc, -1))
        og.submit(res["pred_pose"][:, :, N_ITER - N_COUNTED:])
        store = og.wait()
        all_sums = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(all_sums, mine)
        got = torch.stack([parallel.scene_checksums(store[0, r].reshape(n_sc, -1)) for r in range(world)])
        gather_ok = bool(torch.equal(got, torch.stack(all_sums))) and int(got.unique().numel()) == world * n_sc
        assert gather_ok, "gathered trajectories do not match their source ranks' checksums"

    for _ in range(args.warmup):
        loop_step()
    l0 = ops.LAUNCHES
    with ClockSampler(local) as cs:
        t_loop = timed(loop_step, args.steps)
    launches = args.steps * eng.graph_steps * eng.launches_per_step + (ops.LAUNCHES - l0)  # graph replays + eager launches
    clocks = cs.summary()
    if args.dump_outputs and rank == 0:
        # eng.results() is what the last eng.run() returned (its buffers are not touched again before e2e below);
        # joint_pose is pred_pose viewed per scene, so it is left out
        res = {k: v for k, v in eng.results().items() if k != "joint_pose"}
        print("dump-outputs:", dump_outputs(args.dump_outputs, {}, res), file=sys.stderr, flush=True)
    units = world * n_sc * args.rollouts * N_COUNTED
    value = units * args.steps / t_loop

    # ---- e2e: host batch in, host trajectories out, scene encoding included, every step
    host_out = torch.empty(n_sc * args.rollouts, batch["sc/ag_valid"].shape[1], N_COUNTED, 3).pin_memory()
    host_valid = torch.empty(n_sc * args.rollouts, batch["sc/ag_valid"].shape[1], N_COUNTED, dtype=torch.bool).pin_memory()

    def e2e_step():
        res = eng.rollout(batch)
        host_out.copy_(res["pred_pose"][:, :, N_ITER - N_COUNTED:], non_blocking=True)
        host_valid.copy_(res["pred_valid"][:, :, N_ITER - N_COUNTED:], non_blocking=True)
        torch.cuda.current_stream().synchronize()

    e2e_step()
    t_e2e = timed(e2e_step, max(1, args.steps))
    e2e = dict(value=units * max(1, args.steps) / t_e2e, unit=UNIT, h2d_bytes_per_step=h2d,
               d2h_bytes_per_step=host_out.numel() * 4 + host_valid.numel())

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        roof_sel, roof_proj, roof = attention_roofline(eng, peaks)
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=t_loop / args.steps * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f32" if args.precision == 0 else "tf32+fp16", data="synthetic",
                    config=dict(workload=f"config 3: closed-loop WOSAC rollout, {n_sc} scenes x {args.rollouts} rollouts "
                                         f"per GPU, 128 agents, 1024 polylines x 20, 40 TL, 11-step history, 90 policy "
                                         f"iterations (80 counted)", scenes_per_gpu=n_sc, rollouts=args.rollouts,
                                policy_iterations=N_ITER, counted_steps=N_COUNTED, rule_checks=bool(args.rule_checks),
                                l2="per-iteration working set (>1 GB of activations) exceeds the 126 MB L2; no flush",
                                launches_per_policy_iteration=eng.launches_per_step, gather_verified=gather_ok,
                                agent_slots=(f"{eng._st['A']} of {eng._A_full} per scene: slots without a valid ground-truth step can never "
                                             f"become valid and are dropped for the rollout, results scattered back "
                                             f"(DESIGN.md 6)" if eng._perm is not None else f"{eng._A_full} (no padding dropped)"),
                                warm_start_dedup=f"encoders of the {eng._s0} teacher-forced (rollout-invariant) leading steps "
                                                 f"run once per scene as one batch, inside the timed loop; steps "
                                                 f"{eng._s0 + 1}..{N_ITER} per rollout (DESIGN.md 6)" if eng._s0 else "off"),
                    clocks=clocks, e2e=e2e, gpu_launches=launches, roofline=roof, roofline_select=roof_sel,
                    roofline_projection=roof_proj)
    if rank == 0 and world == 1 and not args.rule_checks and not args.no_extras:
        # extra lines (not the headline): fp32-parity projections, and the loop with ALL TrafficRuleChecker checks on
        extras = {}
        for name, kw in (("fp32_projections", dict(precision=0)), ("fp32_projections_ffma", dict(precision=0)),
                         ("with_rule_checks", dict(precision=args.precision, rule_checks=True))):
            del eng
            torch.cuda.empty_cache()
            eng = RolloutEngine(P, cfg, dev, n_rollout=args.rollouts, step_end=N_ITER, **kw)
            eng.model.fp32_tc = name != "fp32_projections_ffma"  # strict-parity mode: 3xTF32 on tcgen05 vs the FFMA kernel
            eng.prepare(batch)
            eng.run()
            eng.run()
            t = timed(eng.run, 3)
            extras[name] = dict(value=units * 3 / t, unit=UNIT, ms_per_step=t / 3 * 1e3)
        # the once-per-scene step before the loop (SURVEY 8(f) rank 3): destination classifier over all polylines
        Pn = params.init_params(cfg, 0, with_navi_predictor=True)
        del eng
        torch.cuda.empty_cache()
        eng = RolloutEngine(Pn, cfg, dev, n_rollout=args.rollouts, step_end=N_ITER, precision=args.precision, use_graph=False)
        mp = eng.encode_scenes(batch)["mp"]
        eng.predict_destinations(batch, mp=mp)
        t = timed(lambda: eng.predict_destinations(batch, mp=mp), 3) / 3
        extras["navi_predictor"] = dict(value=t * 1e3, unit="ms per batch of scenes (destination logits + sampling, map tokens given)",
                                        scenes=args.scenes)
        del eng
        torch.cuda.empty_cache()
        try:
            extras["knarpe_microbench"] = knarpe_microbench(dev, peaks)
        except Exception as e:
            extras["knarpe_microbench"] = dict(unavailable=f"{type(e).__name__}: {e}"[:200])
        # the real bar: reference-order eager PyTorch on this same GPU (fp32 and fp16 autocast)
        for name, ac in (("eager_cuda_fp32", False), ("eager_cuda_fp16_autocast", True)):
            try:
                extras[name] = eager_cuda_rate(dev, n_sc, args.rollouts, 20, ac)
            except Exception as e:  # a baseline leg must never take the headline line down
                extras[name] = dict(unavailable=f"{type(e).__name__}: {e}"[:200])
        line["extras"] = extras
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        rate, sample, _ = cpu_rollout_rate(cores, 1, 16, 16)
        line["cpu_baseline"] = dict(value=rate, unit=UNIT, cores=cores, kind="port", sample=sample)
        try:  # the same with every logging-only TrafficRuleChecker check on (SURVEY 8(d): "with and without")
            rate_rc, sample_rc, _ = cpu_rollout_rate(cores, 1, 8, 6, rule_checks=True)
            line["cpu_baseline"]["with_rule_checks"] = dict(value=rate_rc, sample=sample_rc)
        except Exception as e:  # a side leg must never take the line down
            line["cpu_baseline"]["with_rule_checks"] = dict(unavailable=f"{type(e).__name__}: {e}"[:200])
    if rank == 0:
        print(json.dumps(line), file=_OUT, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_train(args):
    """BASELINE config 4: forward + backward of the training_step body (waymo_motion.py:313-385) at --scenes scenes of
    the config-3 shape, dropout 0, fp32 rows with tf32 tcgen05 GEMMs (--precision 1) or fp32 FFMA (0). Unit: training
    scene-steps/s = scenes x 90 policy iterations / time of one loss + gradient evaluation. Side numbers: the same step
    by torch autograd through the reference-order oracle on this GPU (`eager_cuda`, a smaller batch: its [B,S,K,2d]
    gathers of all 90 steps do not fit otherwise) and the gradient check against it."""
    import torch.distributed as dist
    from trafficbotsv1_5_b200 import ops
    from trafficbotsv1_5_b200.training import TRAIN_CFG, TrainStep
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: there is no CPU fallback for the product path"
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    cfg = config.default_model_cfg()
    P = params.init_params(cfg, 0, with_navi_predictor=True, with_latent_post=True)
    n_sc = args.scenes if args.scenes != 16 else 64
    batch = synth.make_train_batch(n_sc, seed=3000 + rank * n_sc)  # data parallel: every rank its own scenes
    batch = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in batch.items()}
    ts = TrainStep(P, cfg, dev, precision=min(args.precision, 1))
    if world > 1:
        ts.data_parallel()  # gradients averaged with one NCCL all-reduce per step (inside the timed region)

    last = {}

    def step():
        ts.zero_grad()
        out = ts.step(batch)
        if args.dump_outputs:
            last["out"] = out
        return float(out["loss"].detach())  # device -> host read of the step's result

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(1, args.warmup)):
        loss = step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    l0 = ops.LAUNCHES
    with ClockSampler(local) as cs:
        e0.record()
        for _ in range(args.steps):
            loss = step()
        e1.record()
        barrier()
    tt = torch.tensor([e0.elapsed_time(e1) * 1e-3 / args.steps], device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t = float(tt)
    phases = ts.timings_ms()
    peak_gb = torch.cuda.max_memory_allocated() / 2 ** 30
    if args.dump_outputs and rank == 0:  # the last step's losses and trajectories, and the gradients it left
        out = last["out"]
        whole = {k: v for k, v in out.items() if torch.is_tensor(v) and k not in ("pred_pose", "pred_valid")}
        whole.update({f"grad.{k}": p.grad for k, p in ts.params.items() if p.grad is not None})
        rows = dict(pred_pose=out["pred_pose"], pred_valid=out["pred_valid"])
        print("dump-outputs:", dump_outputs(args.dump_outputs, whole, rows), file=sys.stderr, flush=True)
    if rank != 0:
        dist.barrier()
        dist.destroy_process_group()
        return
    line = dict(metric="training_step_scene_steps_per_sec", value=world * n_sc * N_ITER / t, unit="scene-steps/s (fwd+bwd)",
                n_gpus=world, steps=args.steps, warmup=args.warmup, ms_per_step=t * 1e3, higher_is_better=True,
                scaling="weak", vs_baseline=None, dtype="f32" if args.precision == 0 else "tf32", data="synthetic",
                config=dict(workload=f"config 4: training_step body fwd+bwd, {n_sc} scenes per GPU, 128 agents, 1024 polylines "
                                     f"x 20, 40 TL, 90 teacher-forced policy iterations, dropout 0"
                                     + (", gradients averaged over the ranks (one NCCL all-reduce)" if world > 1 else ""),
                            scenes_per_gpu=n_sc,
                            l2="activations of 90 steps (tens of GB) exceed the 126 MB L2; no flush"),
                clocks=cs.summary(), gpu_launches=ops.LAUNCHES - l0, loss=loss, peak_hbm_gib=peak_gb, phases_ms=phases,
                e2e=dict(value=world * n_sc * N_ITER / t, unit="scene-steps/s (fwd+bwd)",
                         h2d_bytes_per_step=sum(v.numel() * v.element_size() for v in batch.values() if torch.is_tensor(v)),
                         d2h_bytes_per_step=4))
    if not args.no_extras and world == 1:
        try:
            from oracle import tb_oracle_train as OT
            n_e = 2
            be = synth.make_train_batch(n_e, seed=3000)
            be = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in be.items()}
            torch.set_default_device(dev)
            try:
                Pg = {k: v.to(dev).requires_grad_(True) for k, v in P.items()}

                def eager():
                    for p_ in Pg.values():
                        p_.grad = None
                    o = OT.training_step(Pg, cfg, config.derived_sizes(cfg), config.DYNAMICS_CFG, TRAIN_CFG, be)
                    o["loss"].backward()
                    return float(o["loss"])

                eager()
                torch.cuda.synchronize()
                t0 = time.time()
                eager()
                torch.cuda.synchronize()
                te = time.time() - t0
            finally:
                torch.set_default_device("cpu")
            line["eager_cuda"] = dict(value=n_e * N_ITER / te, unit="scene-steps/s (fwd+bwd)", scenes=n_e,
                                      note="torch autograd through the reference-order oracle on this GPU, fp32")
        except Exception as e:
            line["eager_cuda"] = dict(unavailable=f"{type(e).__name__}: {e}"[:200])
    print(json.dumps(line), file=_OUT, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


_OUT = sys.stdout


def _reserve_stdout():
    """stdout carries exactly one JSON line: anything a library prints to fd 1 (NCCL's version banner under torchrun)
    goes to stderr instead, and the line itself is written to the original descriptor (_OUT)."""
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


if __name__ == "__main__":
    a = parse()
    _reserve_stdout()
    if a.impl == "reference":
        run_reference(a)
    elif a.train:
        run_train(a)
    elif a.scenes_total > 0:
        run_sweep(a)
    else:
        run_ours(a)
