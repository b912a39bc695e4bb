"""CPU reference of caller control in the closed loop, built from `oracle/tb_oracle.py`'s pieces: the player override
of Dynamics.update_ag (utils/dynamics.py:96-99), `rollout(..., player_policy)` (pl_modules/waymo_motion.py:206-217) and
whole-agent teacher forcing (utils/teacher_forcing.py:87-92, `tb_oracle_train.teacher_forcing_mask_training`).
With `player=None, forcing_agent=None` `rollout` is `tb_oracle.rollout` (checked by tests/test_player_control_cpu.py)."""
from typing import Dict, Optional

import torch
import torch.nn.functional as F
from torch import Tensor

from oracle import tb_oracle as O
from oracle.tb_oracle_train import teacher_forcing_mask_training


def dynamics_update(pose, motion, valid, ag_type, mean, dyn, player_valid: Optional[Tensor] = None,
                    player_action: Optional[Tensor] = None):
    """`tb_oracle.dynamics_update` with the player override: for valid agents with `player_valid` [B, A] set, the
    physical `player_action` [B, A, 2] (acc m/s^2, yaw rate rad/s) replaces the tanh-scaled action (dynamics.py:96-99),
    before the unicycle update. Agents without a type still come out as zeros."""
    dt = dyn["dt"]
    th = torch.tanh(mean)
    action = 0
    for i, k in enumerate(("veh", "ped", "cyc")):
        a = torch.stack([th[..., 0] * dyn[k]["max_acc"], th[..., 1] * dyn[k]["max_yaw_rate"]], -1)
        action = action + a.masked_fill(~ag_type[:, :, [i]], 0.0)
    action = action.masked_fill(~valid.unsqueeze(-1), 0.0)
    if player_valid is not None:
        action = torch.where((player_valid & valid).unsqueeze(-1), player_action.to(action.dtype), action)
    acc, yr = action[..., 0], action[..., 1]
    v_t = motion[..., 0] + 0.5 * dt * acc
    th_t = pose[..., 2] + 0.5 * dt * yr
    new_pose = pose + dt * torch.stack([v_t * th_t.cos(), v_t * th_t.sin(), yr], -1)
    new_motion = torch.stack([motion[..., 0] + dt * acc, acc, yr], -1)
    keep = valid.unsqueeze(-1) & ag_type.any(-1, keepdim=True)
    return new_pose.masked_fill(~keep, 0.0), new_motion.masked_fill(~keep, 0.0)


def rollout(P, cfg, sz, dyn, rcfg, batch: Dict[str, Tensor], n_rollout: int, step_end: Optional[int] = None,
            player=None, forcing_agent: Optional[Tensor] = None) -> Dict[str, Tensor]:
    """`tb_oracle.rollout` (no rule checks) with caller control:
    player: callable (step, valid, pose, motion) -> (player_valid [n_sc*R, A] bool, action [n_sc*R, A, 2]), called
      every step with the state at time step - 1 (the policy's input), the reference's player_policy hook;
    forcing_agent [n_sc, A] bool: these agents are teacher-forced wherever their ground truth is valid (log replay)."""
    R = n_rollout
    step_end = rcfg["time_step_end"] if step_end is None else step_end
    mp = O.map_encoder(P, cfg, sz, batch["sc/mp_valid"], batch["sc/mp_attr"], batch["sc/mp_pose"])
    tl = O.tl_pre_compute(P, cfg, sz, batch["sc/tl_valid"], batch["sc/tl_attr"], batch["sc/tl_pose"], mp)
    rep = lambda t: t.repeat_interleave(R, 0)  # noqa: E731
    mpR = {k: rep(v) for k, v in mp.items()}
    tlR = {k: rep(v) for k, v in tl.items()}
    gt_valid, gt_pose, gt_motion = rep(batch["sc/ag_valid"]), rep(batch["sc/ag_pose"]), rep(batch["sc/ag_motion"])
    ag_attr, ag_type = rep(batch["sc/ag_attr"]), rep(batch["ref/ag_type"])
    tl_gt = rep(batch["sc/tl_state"])
    n_sc = batch["sc/ag_valid"].shape[0]
    latent = batch["ag_latent"][:, :R].reshape(n_sc * R, *batch["ag_latent"].shape[2:])
    latent_valid = rep(batch["ag_latent_valid"])
    navi, navi_valid = rep(batch["agent/dest"]), rep(batch["ag_navi_valid"]).clone()
    boundary = rep(batch["map/boundary"])
    dest = O.dest_tables(rep(batch["map/valid"]), rep(batch["map/type"]), rep(batch["map/pos"][..., :2]),
                         rep(batch["map/dir"][..., :2]), navi)
    dest_reached = torch.zeros_like(navi_valid)
    tf = teacher_forcing_mask_training(gt_valid, rcfg["step_spawn_agent"], rcfg["step_warm_start"],
                                       None if forcing_agent is None else rep(forcing_agent))
    n_gt = gt_valid.shape[-1]
    valid, pose, motion = gt_valid[:, :, 0], gt_pose[:, :, 0], gt_motion[:, :, 0]
    disabled = torch.zeros_like(valid)
    tl_state = tl_gt[:, :, 0]
    policy = O.PolicyOracle(P, cfg, sz)
    out = dict(pred_valid=[], pred_pose=[], pred_motion=[], tl_state=[])
    for step in range(1, step_end + 1):
        mean, logits = policy.step(valid, pose, motion, ag_attr, ag_type, latent, latent_valid, navi, navi_valid,
                                   tl_state, tlR, mpR)
        pv = pa = None
        if player is not None:
            pv, pa = player(step, valid, pose, motion)
        pred_valid = valid
        pose, motion = dynamics_update(pose, motion, valid, ag_type, mean, dyn, pv, pa)
        pred_pose, pred_motion = pose, motion
        if step < n_gt:
            ov = tf[:, :, step] & ~disabled
            valid = valid | ov
            pose = torch.where(ov.unsqueeze(-1), gt_pose[:, :, step], pose)
            motion = torch.where(ov.unsqueeze(-1), gt_motion[:, :, step], motion)
        tl_new = F.one_hot(torch.softmax(logits, -1).argmax(-1), logits.shape[-1]).bool()
        tl_state = tl_gt[:, :, step] if step < n_gt else tl_new
        outside = O.check_outside_map(pred_valid, pred_pose, boundary)
        reached = O.check_dest_reached(pred_valid, pred_pose, dest, dest_reached)
        dest_reached = dest_reached | reached
        out["pred_valid"].append(pred_valid); out["pred_pose"].append(pred_pose)
        out["pred_motion"].append(pred_motion); out["tl_state"].append(tl_state)
        mask_dis = outside & ~gt_valid[:, :, step] if step < n_gt else outside
        disabled = disabled | mask_dis
        valid = valid & ~mask_dis
        navi_valid = navi_valid & ~reached
    res = {k: torch.stack(v, 2) for k, v in out.items()}
    res["final_valid"], res["final_navi_valid"] = valid, navi_valid
    return res
