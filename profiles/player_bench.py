"""Cost of caller control at BASELINE config 3 (16 scenes x 32 rollouts, 128 agents, 1024 polylines x 20, 40 TL, 90
policy iterations, tensor-core mode), in one process, modes alternating round by round:
  default  RolloutEngine.run() without player keys (what bench.py times);
  plan     run() with an open-loop plan for one agent per rollout ("player/valid" + "player/action");
  stepwise begin() (untimed) + one step() per remaining policy iteration with a trivial controller on the device
           (acc = -0.5 v), i.e. one host round trip per step: reported as host overhead per step against the graph
           replays of `plan` (run() minus run(S0), the warm-start block).
Prints one JSON object (and writes it to --out): card name and power limit are read in the same run.

    python profiles/player_bench.py --rounds 5 --runs 3 --out /tmp/player_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import tbpkg  # noqa: E402,F401
from trafficbotsv1_5_b200 import config, params, synth  # noqa: E402
from trafficbotsv1_5_b200.engine import RolloutEngine  # noqa: E402

N_ITER, N_COUNTED = 90, 80


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
    except Exception as e:  # the number is still a measurement; say what is missing
        out = f"nvidia-smi unavailable: {e}"
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=16)
    ap.add_argument("--rollouts", type=int, default=32)
    ap.add_argument("--precision", type=int, default=1)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--runs", type=int, default=3, help="timed calls per mode and round")
    ap.add_argument("--out")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "player_bench.py needs a CUDA device"
    torch.cuda.set_device(0)
    n_sc, R = args.scenes, args.rollouts
    cfg = config.default_model_cfg()
    eng = RolloutEngine(params.init_params(cfg, 0), cfg, "cuda:0", precision=args.precision, n_rollout=R,
                        step_end=N_ITER)
    batch = synth.make_scene_batch(n_sc=n_sc, seed=1000, n_rollout=R)
    A = batch["sc/ag_valid"].shape[1]
    first = batch["sc/ag_valid"][:, :, 0].float().argmax(1)           # one player per rollout: a valid agent
    pv = torch.zeros(n_sc, A, dtype=torch.bool)
    pv[torch.arange(n_sc), first] = True
    t = torch.arange(N_ITER, dtype=torch.float32)
    amp = torch.linspace(-2.0, 2.0, R)[None, :, None, None]
    pa = torch.stack([amp * torch.cos(0.1 * t).expand(n_sc, R, A, -1), 0.05 * torch.sin(0.1 * t).expand(n_sc, R, A, -1)], -1)
    plan_batch = dict(batch, **{"player/valid": pv, "player/action": pa})
    step_batch = dict(batch, **{"player/valid": pv})

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        h0 = time.perf_counter()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3, time.perf_counter() - h0

    def stepwise():
        obs = eng._observe()
        while obs["t"] < N_ITER:
            v = obs["motion"][..., 0].view(n_sc, R, A)
            obs = eng.step(torch.stack([-0.5 * v, torch.zeros_like(v)], -1))
        return obs

    # default / plan: whole run() (reset, warm-start block, graph replays); plan_warm: run(S0), the part before the
    # graph replays; stepwise: the step() loop after begin() (begin itself is not timed)
    eng.prepare(batch)
    s0 = eng._s0
    modes = {"default": (batch, eng.run), "plan": (plan_batch, eng.run),
             "plan_warm": (plan_batch, lambda: eng.run(s0)), "stepwise": (step_batch, stepwise)}

    def setup(k, b):
        if k == "stepwise":
            eng.begin(b)
        else:
            eng.prepare(b)

    for k, (b, fn) in modes.items():  # warm-up: graphs of both player modes, allocator, lazy module loads
        setup(k, b)
        fn()
    times = {k: [] for k in modes}
    for _ in range(args.rounds):
        for k, (b, fn) in modes.items():
            for _ in range(args.runs):
                setup(k, b)
                times[k].append(timed(fn)[0])
    n_stepped = N_ITER - s0                                            # steps that go through step() / graph replays
    units = n_sc * R * N_COUNTED
    res = {k: dict(s_per_call=sorted(v), median_s=sorted(v)[len(v) // 2]) for k, v in times.items()}
    for k in ("default", "plan"):
        res[k]["rollout_scene_steps_per_s"] = units / res[k]["median_s"]
    replay_us = (res["plan"]["median_s"] - res["plan_warm"]["median_s"]) / n_stepped * 1e6
    res["plan"]["graph_step_us"] = replay_us
    res["stepwise"]["step_us"] = res["stepwise"]["median_s"] / n_stepped * 1e6
    res["stepwise"]["host_overhead_per_step_us"] = res["stepwise"]["step_us"] - replay_us
    res["plan"]["vs_default"] = res["plan"]["median_s"] / res["default"]["median_s"] - 1
    spread = {k: (max(v) - min(v)) / min(v) for k, v in times.items()}
    out = dict(card=card(), workload=f"config 3: {n_sc} scenes x {R} rollouts, 128 agents, 1024 polylines x 20, 40 TL, "
                                     f"{N_ITER} policy iterations ({N_COUNTED} counted), precision={args.precision}",
               players="one agent per rollout (plan / controller)", rounds=args.rounds, runs_per_round=args.runs,
               warm_start_steps=eng._s0, stepped_steps=n_stepped, modes=res, spread_max_over_min=spread)
    line = json.dumps(out, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
