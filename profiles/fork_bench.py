"""Cost of snapshot / restore / fork of the rollout engine at BASELINE config 3 (16 scenes x 32 rollouts, 128 agents,
1024 polylines x 20, 40 TL, 90 policy iterations, tensor-core mode), one player agent per rollout:
  copies    snapshot(), restore(), restore(snap, src) with a fork map: bytes of the state (from the buffer shapes),
            time per call (CUDA events over many calls) and the achieved rate (bytes read + written over time); the same
            copies as one tb_copy_rows launch alone, and as a per-buffer torch copy_ / index_select loop (kept in this
            script only, as the yardstick of the one-launch kernel);
  planning  a receding-horizon loop (H steps of R candidate plans, score, restore + fork, commit one step) against
            the loop it replaces (begin() and a replay of the t committed steps every cycle).
Prints one JSON object (and writes it to --out); the card's name and power limit are read in the same run.

    python profiles/fork_bench.py --out profiles/r3/fork_bench.json
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import tbpkg  # noqa: E402,F401
from trafficbotsv1_5_b200 import config, ops, params, synth  # noqa: E402
from trafficbotsv1_5_b200.engine import RolloutEngine  # noqa: E402
from player_bench import card  # noqa: E402

N_ITER = 90


def events_ms(fn, n):
    """Mean device time of fn() over n back-to-back calls (CUDA events), after one warm-up call."""
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=16)
    ap.add_argument("--rollouts", type=int, default=32)
    ap.add_argument("--precision", type=int, default=1)
    ap.add_argument("--calls", type=int, default=200, help="timed copies per variant")
    ap.add_argument("--horizon", type=int, default=10)
    ap.add_argument("--cycles", type=int, default=20)
    ap.add_argument("--out")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "fork_bench.py needs a CUDA device"
    torch.cuda.set_device(0)
    n_sc, R, H = args.scenes, args.rollouts, args.horizon
    cfg = config.default_model_cfg()
    eng = RolloutEngine(params.init_params(cfg, 0), cfg, "cuda:0", precision=args.precision, n_rollout=R,
                        step_end=N_ITER)
    batch = synth.make_scene_batch(n_sc=n_sc, seed=1000, n_rollout=R)
    A = batch["sc/ag_valid"].shape[1]
    first = batch["sc/ag_valid"][:, :, 0].float().argmax(1)            # one player per rollout: a valid agent
    pv = torch.zeros(n_sc, A, dtype=torch.bool)
    pv[torch.arange(n_sc), first] = True
    b = dict(batch, **{"player/valid": pv})
    g = torch.Generator(device="cuda").manual_seed(0)

    # ------------------------------------------------------------------------------------------ copies
    s0 = eng.begin(b)["t"]
    for _ in range(20):
        eng.step()
    snap = eng.snapshot()
    nbytes = snap.nbytes
    items = eng._state_items()
    fork = torch.randint(0, R, (n_sc, R), generator=g, device="cuda")
    fork_cpu = fork.cpu()
    fork_dev = fork.to(torch.int32).reshape(-1)
    rows = (torch.arange(n_sc, device="cuda")[:, None] * R + fork).reshape(-1)
    dst = [(t, snap._bufs[k], pr) for k, t, pr in items]

    def torch_copy(gather):
        for t, s, pr in dst:
            if gather and pr:
                torch.index_select(s, 0, rows, out=t)
            else:
                t.copy_(s)

    variants = {
        "snapshot": lambda: eng.snapshot(),
        "restore": lambda: eng.restore(snap),
        "restore_fork": lambda: eng.restore(snap, fork_cpu),
        "kernel_copy": lambda: ops.copy_rows([(s, t, pr) for t, s, pr in dst], None, R),
        "kernel_fork": lambda: ops.copy_rows([(s, t, pr) for t, s, pr in dst], fork_dev, R),
        "torch_copy": lambda: torch_copy(False),
        "torch_fork": lambda: torch_copy(True),
    }
    copies = {}
    for rnd in range(2):  # two passes, interleaved: the second is reported, the first shows the spread
        for k, fn in variants.items():
            ms = events_ms(fn, args.calls)
            copies.setdefault(k, {})[f"pass{rnd}_ms"] = ms
    for k, v in copies.items():
        v["ms"] = v["pass1_ms"]
        v["GB_per_s_read_plus_write"] = 2 * nbytes / (v["ms"] * 1e-3) / 1e9
    per_buffer = {k: t.numel() * t.element_size() for k, t, _ in items}

    # ------------------------------------------------------------------------------------------ planning loop
    T = eng.T
    amp = torch.linspace(-2.0, 2.0, R, device="cuda")
    cands = torch.zeros(n_sc, R, A, H, 2, device="cuda")
    cands[..., 0] = amp[None, :, None, None]                           # candidate r: constant acceleration amp[r]
    player = pv.to("cuda")

    def cost():
        x = eng.results()["pred_pose"][..., 0].view(n_sc, R, A, T)      # progress along x of the player, to be maximised
        t = eng._t
        return -(x[:, :, :, t - 1] * player[:, None]).sum(-1)

    def cycle_fork():
        snap_c = eng.snapshot()
        for h in range(H):
            eng.step(cands[:, :, :, h])
        best = cost().argmin(1)
        e_r0.record()
        eng.restore(snap_c, torch.zeros_like(best)[:, None].expand(-1, R))
        e_r1.record()
        return eng.step(cands[torch.arange(n_sc), best][:, None, :, 0].expand(-1, R, -1, -1))

    def cycle_replay(committed):
        """The same cycle without snapshots: begin(), replay the committed steps, H candidate steps, score; the
        chosen first action is committed by the next cycle's replay."""
        eng.begin(b)
        for c in committed:
            eng.step(c)
        for h in range(H):
            eng.step(cands[:, :, :, h])
        best = cost().argmin(1)
        return cands[torch.arange(n_sc), best][:, None, :, 0].expand(-1, R, -1, -1)

    loops = {}
    for rnd in range(2):  # first pass: warm-up (graphs, allocator)
        e_r0, e_r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        eng.begin(b)
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        restore_ms = 0.0
        for _ in range(args.cycles):
            cycle_fork()
            torch.cuda.synchronize()
            restore_ms += e_r0.elapsed_time(e_r1)
        fork_s = time.perf_counter() - h0
        t_end = eng._t
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        committed = []
        for c in range(args.cycles):
            committed.append(cycle_replay(committed))
        torch.cuda.synchronize()
        replay_s = time.perf_counter() - h0
        loops = dict(cycles=args.cycles, horizon=H, candidates=R, t_start=s0, t_end=t_end,
                     fork_ms_per_cycle=fork_s / args.cycles * 1e3,
                     restore_call_ms_per_cycle=restore_ms / args.cycles,
                     snapshot_ms_per_cycle=copies["snapshot"]["ms"],
                     replay_ms_per_cycle=replay_s / args.cycles * 1e3)
    loops["snapshot_restore_share"] = (loops["snapshot_ms_per_cycle"] + loops["restore_call_ms_per_cycle"]) / \
        loops["fork_ms_per_cycle"]
    loops["speedup_vs_replay"] = loops["replay_ms_per_cycle"] / loops["fork_ms_per_cycle"]

    out = dict(card=card(), workload=f"config 3: {n_sc} scenes x {R} rollouts, 128 agents, 1024 polylines x 20, 40 TL, "
                                     f"{N_ITER} policy iterations, precision={args.precision}, one player per rollout",
               state_bytes=nbytes, state_buffers=len(items), per_buffer_bytes=per_buffer, calls_per_variant=args.calls,
               copies=copies, receding_horizon=loops,
               notes="ms per call: CUDA events over back-to-back calls of the same copy (a %.0f MB state, each copy "
                     "reads and writes it: no L2 flush between calls); planning loop: host clock with a device "
                     "synchronise per cycle" % (nbytes / 1e6))
    line = json.dumps(out, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
