"""Closed-loop WOSAC rollout engine: the reference's `WaymoMotion.test_step -> joint_future_pred -> rollout ->
forward` chain (src/pl_modules/waymo_motion.py:843-876, 439-524, 206-311, 118-204) on the CUDA hot path.

Differences in HOW (not WHAT), see DESIGN.md §4:
  * the 32 rollouts of a scene index the scene's map / traffic-light tables (`b // R`) instead of
    `repeat_interleave` copies (:458-462);
  * the traffic-light branch depends only on (scene, TL history) — identical across a scene's rollouts and
    deterministic (argmax, dynamics.py:154-159) — so it is evaluated once per scene (`tl_per_scene`);
  * rollout state, history rings and the trajectory buffers stay resident in HBM for all steps; the loop counter
    is a device scalar, so ONE captured CUDA graph is replayed for every step with no host sync.
"""
from typing import Dict, Optional

import numpy as np
import torch
from torch import Tensor

from . import config as C
from . import lib as L
from . import ops
from .model import HotPathModel


VIOLATIONS = ("collided", "collided_wosac", "run_road_edge", "run_red_light", "passive")


def rule_tables(mp_valid: Tensor, mp_type: Tensor, mp_pos: Tensor, mp_dir: Tensor) -> Dict[str, Tensor]:
    """Per-scene map tables for tb_rule_check (TrafficRuleChecker._get_road_edge / _get_lane_center,
    utils/traffic_rule_checker.py:452-497): segments (pos, pos + dir), node validity, a bounding circle per polyline
    and its kind bits (1: road-edge types 4,5,7; 2: lane-centre types 0..2)."""
    end = mp_pos + mp_dir
    seg = torch.cat([mp_pos, end], -1).contiguous()                                     # [n_sc, n_mp, n_node, 4]
    pts = torch.cat([mp_pos, end], 2)                                                   # [n_sc, n_mp, 2*n_node, 2]
    centre = 0.5 * (pts.amin(2) + pts.amax(2))
    radius = torch.norm(pts - centre[:, :, None], dim=-1).amax(2) + 1e-3
    kind = mp_type[:, :, [4, 5, 7]].any(-1).to(torch.uint8) + 2 * mp_type[:, :, :3].any(-1).to(torch.uint8)
    return dict(seg=seg, node_invalid=(~mp_valid).to(torch.uint8).contiguous(),
                poly_circle=torch.cat([centre, radius[..., None]], -1).contiguous(), poly_kind=kind.contiguous())


def teacher_forcing_mask(gt_valid: Tensor, step_spawn: int, step_warm: int) -> Tensor:
    """TeacherForcing.init at test time (utils/teacher_forcing.py:51-82; schedules / thresholds off)."""
    tf = torch.zeros_like(gt_valid)
    tf[:, :, 0] |= gt_valid[:, :, 0]
    if step_spawn > 0:
        spawn = (~gt_valid[:, :, :-1]) & gt_valid[:, :, 1:]
        spawn[:, :, step_spawn:] = False
        tf[:, :, 1:] |= spawn
    if step_warm >= 0:
        tf[:, :, : step_warm + 1] |= gt_valid[:, :, : step_warm + 1]
    return tf


def _leaves(tree, out):
    if isinstance(tree, Tensor):
        out.append(tree)
    elif isinstance(tree, dict):
        for k in sorted(tree):
            _leaves(tree[k], out)
    elif isinstance(tree, (list, tuple)):
        for v in tree:
            _leaves(v, out)
    else:
        out.append(tree)
    return out


def _same_layout(a, b) -> bool:
    la, lb = _leaves(a, []), _leaves(b, [])
    if len(la) != len(lb):
        return False
    for x, y in zip(la, lb):
        if isinstance(x, Tensor) != isinstance(y, Tensor):
            return False
        if isinstance(x, Tensor):
            if x.shape != y.shape or x.dtype != y.dtype or x.stride() != y.stride():
                return False
        elif x != y:
            return False
    return True


def _copy_tree(dst, src) -> None:
    """dst <- src leaf by leaf (views that alias one buffer are copied redundantly but consistently)."""
    for x, y in zip(_leaves(dst, []), _leaves(src, [])):
        if isinstance(x, Tensor) and x.data_ptr() != y.data_ptr():
            x.copy_(y)


class RolloutEngine:
    def __init__(self, P: Dict[str, Tensor], cfg: Optional[dict] = None, device="cuda", precision: int = 0,
                 n_rollout: int = 32, step_end: Optional[int] = None, use_graph: bool = True,
                 rule_checks: bool = False, record_feedback: bool = False, dynamics_cfg: Optional[dict] = None):
        L.load()  # fail loudly if the CUDA library is missing
        self.cfg = cfg or C.default_model_cfg()
        self.sz = C.derived_sizes(self.cfg)
        self.dev = torch.device(device)
        self.model = HotPathModel(P, self.cfg, self.sz, device, precision)
        self.R = n_rollout
        self.T = step_end or C.ROLLOUT_CFG["time_step_end"]
        self.tl_per_scene = True  # the TL branch is a function of (scene, TL history) only: evaluated once per scene
        self.use_graph = use_graph
        self.rule_checks = rule_checks  # also evaluate the logging-only TrafficRuleChecker checks every step
        # also keep outside_map_this_step / dest_reached_this_step of every step (RolloutBuffer.violation, buffer.py:57-60)
        self.record_feedback = record_feedback
        self.dyn = dynamics_cfg or C.DYNAMICS_CFG
        # inference teacher forcing (teacher_forcing.py:51-82): spawn up to / warm start up to these steps
        self.tf_steps = (C.ROLLOUT_CFG["step_spawn_agent"], C.ROLLOUT_CFG["step_warm_start"])
        # Warm-start de-duplication: while every valid agent is teacher-forced (steps 1 .. step_warm_start + 1 of a scene
        # without track gaps) the encoder inputs of the R rollouts of a scene are identical and known from the ground
        # truth alone, so the agent / TL encoders of those steps run ONCE per scene, all steps in one batch (_warm_*).
        self.warm_dedup = True
        self._s0 = 0         # number of leading policy steps handled that way for the prepared batch
        # Agent compaction: agents without a single valid ground-truth step can never become valid (spawning needs
        # ground truth, teacher_forcing.py:51-82), so every scene's agents are reordered valid-first and the padding
        # beyond the largest valid count of the batch (rounded up to 4) is dropped for the whole rollout; results()
        # scatters back to the caller's agent order. WOMD scenes are padded to 128 agents, few have that many.
        self.compact_agents = True
        self._perm = None    # [n_sc, A_eff] original agent index of every kept slot (None: nothing dropped)
        self._A_full = 0
        self.graph_steps = 0  # graph replays of the last run() (bench.py: launch accounting)
        self._by_shape = {}  # shape -> (state, static, navi, graphs, launches per step) of recently used batch shapes
        self._static = self._navi = None
        # player mode -> (graph for odd steps, graph for even steps): the TL branch is double-buffered, and a batch with
        # "player/valid" launches the dynamics with the player override (tb_dyn_step_player), so it has graphs of its own
        self._graphs = {}
        self._players = False  # the prepared batch has player-controlled agents
        self._t = None       # current time of step-by-step stepping (begin / step); None: not begun
        self._host_step = 1  # parity source for eager _step calls
        self._shape = None
        self._side = torch.cuda.Stream(device=self.dev)  # traffic-light branch runs beside the agent front-end
        self._side2 = torch.cuda.Stream(device=self.dev)  # KNN selects run beside the history encoder and layer 0
        self._side3 = torch.cuda.Stream(device=self.dev)
        self._sat = ops.fp16_flag(self.dev)  # fp16 range guard of the tensor-core mode (include/tb_knarpe.h)
        # constants rounded the way the reference's fp32 tensor ops round them (traffic_rule_checker.py:94-96,103,308)
        one = torch.ones(1)
        self.thresh_lane = float(one * 50 * (1 - torch.zeros(1) * 0.8))
        self.thresh_edge = float(one * 50 * (1 - one * 0.8))
        self.cos_rot = float(torch.tensor(np.cos(np.deg2rad(30)), dtype=torch.float32))

    @property
    def _graph(self):
        """Step graphs of the prepared batch's shape and player mode (None until captured)."""
        return self._graphs.get(self._players)

    # ---------------------------------------------------------------------------------------------- scene encoding
    def encode_scenes(self, batch: Dict[str, Tensor]) -> dict:
        """Once per scene: map encoder, TL static tokens, per-layer map K/V tables (test_step :847-851)."""
        dev = self.dev
        g = lambda k: batch[k].to(dev)  # noqa: E731
        mp = self.model.map_encoder(g("sc/mp_valid"), g("sc/mp_attr"), g("sc/mp_pose"))
        tl = self.model.tl_pre_compute(g("sc/tl_valid"), g("sc/tl_attr"), g("sc/tl_pose"), mp)
        kv_mp = self.model.ag_static(mp)
        return dict(mp=mp, tl=tl, kv_mp=kv_mp)

    @torch.no_grad()
    def static_from_tokens(self, mp_tokens: Dict[str, Tensor], tl_tokens: Dict[str, Tensor]) -> dict:
        """The `static` argument of `prepare` from per-scene token dicts in the reference's layout, as the `TrafficBots`
        drop-in's `mp_encoder` / `tl_encoder.pre_compute` return them (map_encoder.py:107-113, traffic_light.py:76-154;
        relative poses raw [.., 3], optional `b200_kv_*` per-layer K|V tables): nothing is re-encoded."""
        m, d, W = self.model, self.model.d, self.model.W
        c = lambda t: t.contiguous()  # noqa: E731
        n_sc, n_mp = mp_tokens["mp_token_pose"].shape[:2]
        n_tl = tl_tokens["tl_token_pose"].shape[1]
        tok_pose, tok_inv = c(mp_tokens["mp_token_pose"].float()), c(mp_tokens["mp_token_invalid"])
        mp = dict(mp_token_invalid=tok_inv, mp_token_feature=c(mp_tokens["mp_token_feature"].float()),
                  mp_token_pose=tok_pose, **m.sorted_map(tok_pose, tok_inv))
        kv_dt = torch.float16 if m.kv_half else torch.float32
        n_ag_l, n_tl_l = self.cfg["ag_encoder"]["n_layer_tf"], self.cfg["tl_encoder"]["n_layer_tf"]

        def tables(prefix, n_layer, layer_name):
            keys = [f"{prefix}{i}" for i in range(n_layer)]
            if all(k in mp_tokens or k in tl_tokens for k in keys):
                tabs = [(mp_tokens.get(k) if k in mp_tokens else tl_tokens[k]) for k in keys]
                if all(t.dtype == kv_dt for t in tabs):
                    return [c(t).view(n_sc * n_mp, 2 * d) for t in tabs]
            feat2d = mp["mp_token_feature"].reshape(n_sc * n_mp, d)
            return [m.kv_table(feat2d, f"{layer_name}.{i}", "norm_tgt") for i in range(n_layer)]

        kv_mp = tables("b200_kv_ag_", n_ag_l, "ag_encoder.tf_ag2agmptl.layers")
        kv_tl = tables("b200_kv_tl_", n_tl_l, "tl_encoder.tf_tl2tlmp.layers")
        for k in ("rpe_tl2tl", "rpe_tl2mp"):
            if tl_tokens[k].shape[-1] != 3:
                raise NotImplementedError(f"{k}: pass the raw relative poses [.., 3] of the drop-in's pre_compute (the "
                                          "embedding is evaluated inside the attention kernel)")
        knn = lambda i, v, r: dict(idx=c(tl_tokens[i].to(torch.int32)), inv=c(tl_tokens[v]), rel=c(tl_tokens[r].float()))  # noqa
        if "knn_idx_tl2mp" not in tl_tokens:
            raise NotImplementedError("tl_tokens need knn_idx_tl2mp (indices), not the pre-gathered knn_tgt_tl2mp features")
        c0 = knn("knn_idx_tl2mp", "knn_invalid_tl2mp", "rpe_tl2mp")
        attr = c(tl_tokens["tl_token_attr"].float()).view(n_sc * n_tl, d)
        tl = dict(n_sc=n_sc, n_tl=n_tl, tl_token_invalid=c(tl_tokens["tl_token_invalid"]),
                  tl_token_pose=c(tl_tokens["tl_token_pose"].float()), tl_token_attr=attr,
                  tl_attr_rows=attr.view(n_sc * n_tl, 1, d).expand(-1, W, -1).reshape(-1, d).contiguous(),
                  knn_self=knn("knn_idx_tl2tl", "knn_invalid_tl2tl", "rpe_tl2tl"),
                  cross=[dict(c0, kv0=kv_tl[i], T0=n_mp, div0=1, K0=self.sz["k_tl2mp"]) for i in range(n_tl_l)])
        return dict(mp=mp, tl=tl, kv_mp=kv_mp)

    @torch.no_grad()
    def predict_destinations(self, batch: Dict[str, Tensor], mp: Optional[dict] = None, deterministic_k0: bool = False,
                             generator: Optional[torch.Generator] = None) -> Dict[str, Tensor]:
        """The once-per-scene step right before the loop (waymo_motion.py:469-495, SURVEY 8(f) rank 3): destination
        distribution of every agent over the map polylines (NaviPredictor "dest" mode, needs `navi_predictor.*`
        weights) and one destination per rollout: rollout 0 takes the argmax when `deterministic_k0`
        (`joint_future_pred_deterministic_k0`, default False as in configs/model/sim_agent.yaml:13), the others are
        sampled (DestCategorical.sample, distributions.py:143-159) with torch's multinomial — once per scene, not part
        of the per-step loop.
        Returns logits [n_sc,n_ag,n_mp], probs, dest int64 [n_sc,R,n_ag] (feed as batch["agent/dest"]) and
        navi_valid [n_sc,n_ag] (batch["ag_navi_valid"])."""
        dev = self.dev
        g = lambda k: batch[k].to(dev)  # noqa: E731
        if mp is None:
            mp = self.model.map_encoder(g("sc/mp_valid"), g("sc/mp_attr"), g("sc/mp_pose"))
        logits = self.model.navi_predictor(g("sc/ag_valid"), g("sc/ag_attr"), g("sc/ag_motion"), g("sc/ag_pose"), mp,
                                           g("ref/ag_type"), g("ref/mp_type"))
        probs = torch.softmax(logits, -1)
        n_sc, A, n_mp = probs.shape
        dest = torch.multinomial(probs.reshape(n_sc * A, n_mp), self.R, replacement=True, generator=generator)
        dest = dest.view(n_sc, A, self.R).permute(0, 2, 1).contiguous()
        if deterministic_k0:
            dest[:, 0] = probs.argmax(-1)
        return dict(logits=logits, probs=probs, dest=dest, navi_valid=g("sc/ag_valid").any(-1))

    # ---------------------------------------------------------------------------------------------- state
    def _alloc(self, n_sc: int, A: int, n_tl: int, n_gt: int, n_mp: int, n_node: int):
        dev, R, W, T, d = self.dev, self.R, self.model.W, self.T, self.model.d
        B = n_sc * R
        Bt = n_sc if self.tl_per_scene else B
        z = lambda *s, dt=torch.float32: torch.zeros(*s, dtype=dt, device=dev)  # noqa: E731
        u8 = torch.uint8
        st = dict(B=B, A=A, Bt=Bt, n_sc=n_sc, n_tl=n_tl, n_gt=n_gt, n_mp=n_mp, n_node=n_node,
                  d_step=z(1, dt=torch.int32),
                  valid=z(B, A, dt=u8), disabled=z(B, A, dt=u8), navi_invalid=z(B, A, dt=torch.bool),
                  dest_reached=z(B, A, dt=u8), pose=z(B, A, 3), motion=z(B, A, 3),
                  hist_valid=z(B, A, W, dt=u8), hist_pose=z(B, A, W, 3), hist_motion=z(B, A, W, 3),
                  hist_tl=z(Bt, n_tl, W, 5, dt=u8),
                  ag_attr=z(B, A, 6), ag_type=z(B, A, 3, dt=u8), latent=z(B * A, self.cfg["latent_encoder"]["latent_dim"]),
                  latent_invalid=z(B, A, dt=torch.bool), dest_idx=z(B, A, dt=torch.int32),
                  gt_valid=z(n_sc, A, n_gt, dt=u8), gt_pose=z(n_sc, A, n_gt, 3), gt_motion=z(n_sc, A, n_gt, 3),
                  tf_mask=z(n_sc, A, n_gt, dt=u8), gt_tl=z(Bt, n_tl, n_gt, 5, dt=u8), boundary=z(n_sc, 4),
                  mp_pos=z(n_sc, n_mp, n_node, 2), mp_dirn=z(n_sc, n_mp, n_node, 2),
                  mp_node_invalid=z(n_sc, n_mp, n_node, dt=u8), mp_kind=z(n_sc, n_mp, dt=u8),
                  pred_valid=z(B, A, T, dt=u8), pred_pose=z(B, A, T, 3), pred_motion=z(B, A, T, 3),
                  tl_out=z(Bt, n_tl, T, 5, dt=u8), x_cat=z(B * A, 2 * d),
                  # traffic-light branch, double-buffered by step parity: TL(s+1) is evaluated during iteration s
                  tl_feat=z(2, Bt * n_tl, d), tl_logits=z(2, Bt * n_tl, self.cfg["tl_state_dim"]),
                  kv_tl=[[torch.empty(Bt * n_tl, 2 * d, device=dev,
                                      dtype=torch.float16 if self.model.kv_half else torch.float32)
                          for _ in range(self.cfg["ag_encoder"]["n_layer_tf"])] for _ in range(2)],
                  d_step_tl=z(1, dt=torch.int32),
                  knn_state=z(B, A, 3),  # agent -> map select: (x, y, K-th squared distance) of the previous step
                  knn_state_tl=z(B, A, 3),  # same for the agent -> traffic-light select
                  init_navi_valid=z(B, A, dt=torch.bool))
        if self.record_feedback:
            st.update(fb_outside=z(B, A, T, dt=u8), fb_reached=z(B, A, T, dt=u8), tl_nll=z(Bt, n_tl, T))
        if self.rule_checks:
            st.update(ag_size=z(n_sc, A, 3), passive_counter=z(B, A), seg=z(n_sc, n_mp, n_node, 4),
                      node_invalid=z(n_sc, n_mp, n_node, dt=u8), poly_circle=z(n_sc, n_mp, 3),
                      poly_kind=z(n_sc, n_mp, dt=u8),
                      **{f"vio_{k}": z(B, A, T, dt=u8) for k in VIOLATIONS})
        return st

    def _load_state(self, st: dict, batch: Dict[str, Tensor]):
        """Dynamics.init / TeacherForcing.init / TrafficRuleChecker.__init__ inputs (dynamics.py:29-64,
        teacher_forcing.py:51-82, traffic_rule_checker.py:86-105), replicated R times by index only."""
        dev, R = self.dev, self.R
        g = lambda k: batch[k].to(dev)  # noqa: E731
        rep = lambda t: t.repeat_interleave(R, 0)  # noqa: E731
        rc = C.ROLLOUT_CFG
        n_sc = st["n_sc"]
        gt_valid = g("sc/ag_valid")
        st["gt_valid"].copy_(gt_valid)
        st["gt_pose"].copy_(g("sc/ag_pose"))
        st["gt_motion"].copy_(g("sc/ag_motion"))
        tf = teacher_forcing_mask(gt_valid, *self.tf_steps)
        if "tf/forcing_agent" in batch:  # log replay of whole agents (teacher_forcing.py:87-92, as TrainStep)
            tf = tf | (g("tf/forcing_agent")[:, :, None] & gt_valid)
        st["tf_mask"].copy_(tf)
        if "player/valid" in batch:  # [n_sc, R, A(, T, 2)] after _player_inputs / _compact
            B, A = st["B"], st["A"]
            if "player_valid" not in st:  # allocated on first use; the player-mode graphs point at these buffers
                st["player_valid"] = torch.zeros(B, A, dtype=torch.uint8, device=dev)
                st["player_action"] = torch.zeros(B, A, self.T, 2, device=dev)
            st["player_valid"].copy_(g("player/valid").reshape(B, A))
            st["player_action"].copy_(g("player/action").reshape(B, A, self.T, 2))
        tl_gt = g("sc/tl_state")
        st["gt_tl"].copy_(tl_gt if self.tl_per_scene else rep(tl_gt))
        st["boundary"].copy_(g("map/boundary"))
        st["ag_attr"].copy_(rep(g("sc/ag_attr")))
        st["ag_type"].copy_(rep(g("ref/ag_type")))
        lat = g("ag_latent")[:, :R]
        st["latent"].copy_(lat.reshape(n_sc * R * st["A"], -1))
        per_rollout = lambda t: t if t.shape[0] == n_sc * R else rep(t)  # noqa: E731  [n_sc, A] or [n_sc*R, A]
        st["latent_invalid"].copy_(~per_rollout(g("ag_latent_valid")))
        dest = g("agent/dest")
        if dest.dim() == 2:  # one destination per (scene, agent); [n_sc, R, A] = per-rollout samples
            dest = dest[:, None].expand(-1, R, -1)
        st["dest_idx"].copy_(dest.reshape(n_sc * R, -1))
        st["init_navi_valid"].copy_(per_rollout(g("ag_navi_valid")))
        mp_dir = g("map/dir")[..., :2]
        st["mp_pos"].copy_(g("map/pos")[..., :2])
        st["mp_dirn"].copy_(mp_dir / torch.norm(mp_dir, dim=-1, keepdim=True))
        st["mp_node_invalid"].copy_(~g("map/valid"))
        mp_type = g("map/type")
        st["mp_kind"].copy_(mp_type[..., :4].any(-1).to(torch.uint8) + 2 * mp_type[..., 4].to(torch.uint8))
        if self.rule_checks:
            st["ag_size"].copy_(g("ref/ag_size"))
            for k, v in rule_tables(g("map/valid"), mp_type, g("map/pos")[..., :2], mp_dir).items():
                st[k].copy_(v)

    def _reset(self, st: dict, tl_prologue: bool = True):
        """time 0 of the rollout (waymo_motion.py:219-227)."""
        R = self.R
        rep = lambda t: t.repeat_interleave(R, 0)  # noqa: E731
        for k in ("disabled", "dest_reached", "hist_valid", "hist_pose", "hist_motion", "hist_tl", "pred_valid",
                  "pred_pose", "pred_motion", "tl_out") + (("fb_outside", "fb_reached") if self.record_feedback else ()):
            st[k].zero_()
        if self.rule_checks:
            st["passive_counter"].zero_()
            for k in VIOLATIONS:
                st[f"vio_{k}"].zero_()
        st["valid"].copy_(rep(st["gt_valid"][:, :, 0]))
        st["pose"].copy_(rep(st["gt_pose"][:, :, 0]))
        st["motion"].copy_(rep(st["gt_motion"][:, :, 0]))
        st["navi_invalid"].copy_(~st["init_navi_valid"])
        st["hist_valid"][:, :, 0] = st["valid"]
        st["hist_pose"][:, :, 0] = st["pose"]
        st["hist_motion"][:, :, 0] = st["motion"]
        st["hist_tl"][:, :, 0] = st["gt_tl"][:, :, 0]
        st["knn_state"].fill_(float("inf"))
        st["knn_state_tl"].fill_(float("inf"))
        st["d_step"].fill_(1)
        st["d_step_tl"].fill_(1)
        self._host_step = 1
        if tl_prologue:
            # prologue of the TL pipeline: tokens / logits / agent-layer tables of step 1 (buffer set 1 = odd steps)
            self._tl_branch(st, self._static, 1)
            st["d_step_tl"].fill_(2)

    def _tl_branch(self, st: dict, static: dict, dst: int):
        """Traffic-light encoder + state predictor for the step `d_step_tl` points to, into buffer set `dst`."""
        m = self.model
        m.tl_forward(st["hist_tl"], st["d_step_tl"], static["tl"], out_feat=st["tl_feat"][dst],
                     out_logits=st["tl_logits"][dst])
        m.ag_tl_tables(st["tl_feat"][dst], out=st["kv_tl"][dst])

    # ---------------------------------------------------------------------------------------------- one step
    def _step(self, st: dict, static: dict, navi: dict, aux: Optional[dict] = None, parity: Optional[int] = None):
        """One policy iteration s. The traffic-light branch depends only on its own history (its state feedback is
        the argmax of its own logits, dynamics.py:154-159), so it is software-pipelined: while the agents of step s
        are encoded on the main stream, the side stream applies the TL feedback of step s and evaluates the TL
        tokens of step s+1 into the other buffer set. The ~70 tiny TL launches then fill the tails of the large
        agent kernels instead of sitting on the critical path of the first agent cross-attention
        (profiles/r1/timeline_final.txt)."""
        m, lib = self.model, L.load()
        d = m.d
        if parity is None:  # eager call: the host knows the step number
            parity = self._host_step % 2
            self._host_step += 1
        cur, nxt = parity, 1 - parity
        tl_feat, logits = st["tl_feat"][cur], st["tl_logits"][cur]
        main = torch.cuda.current_stream()
        self._side.wait_stream(main)
        with torch.cuda.stream(self._side):
            L.check(lib.tb_tl_step_ex(L.ptr(logits), L.ptr(ops._u8(static["tl"]["tl_token_invalid"])), L.ptr(st["gt_tl"]),
                                      st["n_gt"], L.ptr(st["d_step"]), st["Bt"], st["n_tl"], m.W, self.T,
                                      L.ptr(st["hist_tl"]), L.ptr(st["tl_out"]), L.ptr(st.get("tl_nll")), L.stream()),
                    "tb_tl_step_ex")
            self._tl_branch(st, static, nxt)
        m.ag_forward(st, static["mp"], static["kv_mp"], static["tl"], tl_feat, self.R, out=st["x_cat"][:, :d],
                     aux=aux, knn_stream=self._side2, knn_stream2=self._side3, kv_tl=st["kv_tl"][cur])
        act = m.heads(st["x_cat"], st, navi)
        if aux is not None:
            aux.update(tl_feat=tl_feat, logits=logits, act=act, ag_feat=st["x_cat"][:, :d].clone())
        self._advance(st, static, act, join=self._side)

    def _advance(self, st: dict, static: dict, act: Tensor, join=None) -> None:
        """Dynamics + teacher forcing + feedback checks of the step (tb_dyn_step), the optional logging checks, and the
        loop counters. `join`: stream whose work (TL feedback / next TL tokens) must be done before the step ends."""
        m, lib = self.model, L.load()
        dy = self.dyn
        order = ("veh", "ped", "cyc")
        args = (
            L.ptr(act), L.ptr(st["ag_type"]), ops.host_f3([dy[k]["max_acc"] for k in order]),
            ops.host_f3([dy[k]["max_yaw_rate"] for k in order]), dy["dt"], L.ptr(st["valid"]), L.ptr(st["disabled"]),
            L.ptr(ops._u8(st["navi_invalid"])), L.ptr(st["dest_reached"]), L.ptr(st["pose"]), L.ptr(st["motion"]),
            L.ptr(st["gt_valid"]), L.ptr(st["gt_pose"]), L.ptr(st["gt_motion"]), L.ptr(st["tf_mask"]), st["n_gt"],
            self.R, L.ptr(st["boundary"]), L.ptr(st["dest_idx"]), L.ptr(st["mp_pos"]), L.ptr(st["mp_dirn"]),
            L.ptr(st["mp_node_invalid"]), L.ptr(st["mp_kind"]), st["n_mp"], st["n_node"], self.thresh_lane,
            self.thresh_edge, self.cos_rot, L.ptr(st["d_step"]), st["B"], st["A"], m.W, self.T, L.ptr(st["hist_valid"]),
            L.ptr(st["hist_pose"]), L.ptr(st["hist_motion"]), L.ptr(st["pred_valid"]), L.ptr(st["pred_pose"]),
            L.ptr(st["pred_motion"]), L.ptr(st.get("fb_outside")), L.ptr(st.get("fb_reached")))
        if self._players:  # the player's plan column s-1 replaces the action head of player agents (dynamics.py:96-99)
            L.check(lib.tb_dyn_step_player(*args, L.ptr(st["player_valid"]), L.ptr(st["player_action"]), L.stream()),
                    "tb_dyn_step_player")
        else:
            L.check(lib.tb_dyn_step_ex(*args, L.stream()), "tb_dyn_step_ex")
        if join is not None:
            torch.cuda.current_stream().wait_stream(join)  # TL feedback of this step applied, TL tokens of the next ready
        if self.rule_checks:
            tlp = static["tl"]
            L.check(lib.tb_rule_check(
                L.ptr(st["pred_valid"]), L.ptr(st["pred_pose"]), L.ptr(st["pred_motion"]), L.ptr(st["ag_type"]),
                L.ptr(st["ag_size"]), L.ptr(st["hist_tl"]), L.ptr(ops._u8(tlp["tl_token_invalid"])),
                L.ptr(tlp["tl_token_pose"]), L.ptr(st["seg"]), L.ptr(st["node_invalid"]), L.ptr(st["poly_circle"]),
                L.ptr(st["poly_kind"]), st["n_mp"], st["n_node"], L.ptr(st["passive_counter"]),
                *[L.ptr(st[f"vio_{k}"]) for k in VIOLATIONS], L.ptr(st["d_step"]), st["B"], st["A"], self.T, m.W,
                st["n_tl"], self.R, self.R if self.tl_per_scene else 1, 1.1, L.stream()), "tb_rule_check")  # hist_tl: Bt rows
            ops._count()
        L.check(lib.tb_step_advance(L.ptr(st["d_step"]), L.stream()), "tb_step_advance")
        L.check(lib.tb_step_advance(L.ptr(st["d_step_tl"]), L.stream()), "tb_step_advance")
        ops._count(4)

    # ---------------------------------------------------------------------------------------------- warm-start de-duplication
    def _invariant_steps(self, st: dict) -> int:
        """Number S0 of leading policy steps whose encoder inputs do not depend on the rollout: the state at time t is
        rollout-invariant while every agent that was valid before t is teacher-forced at t (then state(t) = ground truth
        where tf[t], invalid elsewhere; such agents are never disabled: their ground truth is valid, dynamics.py:176-178).
        Step s reads times < s, so steps 1 .. t_inv + 1 qualify. One host read per prepared batch."""
        tf = st["tf_mask"].bool()                                    # [n_sc, A, n_gt]
        v_prev = torch.cummax(tf.to(torch.uint8), 2)[0].bool()[:, :, :-1]
        ok = (tf[:, :, 1:] | ~v_prev).all(0).all(0)                  # C(t), t = 1 .. n_gt - 1
        bad = torch.nonzero(~ok)
        t_inv = int(bad[0]) if bad.numel() else ok.numel()           # C(1 .. t_inv) hold
        s0 = min(t_inv + 1, self.T, st["n_gt"])
        return s0 if s0 >= 3 else 0

    def _build_warm(self, st: dict, static: dict) -> dict:
        """History rings of the S0 rollout-invariant steps as a batch of n_sc x S0 rows (scene, step), built from the
        ground truth alone (pure data movement, done at prepare time)."""
        m, dev, R, S0 = self.model, self.dev, self.R, self._s0
        W, d = m.W, m.d
        n_sc, A, n_tl = st["n_sc"], st["A"], st["n_tl"]
        s1 = torch.arange(S0, device=dev)[:, None]
        k = torch.arange(W, device=dev)[None, :]
        t = s1 - torch.remainder(s1 - k, W)                          # ring slot k of step s holds time t (traffic_bots.py:123-143)
        tmask, tidx = t >= 0, t.clamp(min=0)
        tf = st["tf_mask"]                                           # u8 [n_sc, A, n_gt]
        m8 = tmask.to(torch.uint8)
        hv = (tf[:, :, tidx].permute(0, 2, 1, 3) * m8[None, :, None, :]).contiguous()            # [n_sc, S0, A, W]
        keep = hv.bool()[..., None]
        hp = (st["gt_pose"][:, :, tidx].permute(0, 2, 1, 3, 4) * keep).contiguous()
        hm = (st["gt_motion"][:, :, tidx].permute(0, 2, 1, 3, 4) * keep).contiguous()
        Bq = n_sc * S0
        d_rows = torch.arange(1, S0 + 1, dtype=torch.int32, device=dev).repeat(n_sc).contiguous()
        stb = dict(B=Bq, A=A, hist_valid=hv.view(Bq, A, W), hist_pose=hp.view(Bq, A, W, 3), hist_motion=hm.view(Bq, A, W, 3),
                   d_step=d_rows, ag_attr=st["ag_attr"][::R].reshape(n_sc, 1, A, 6).expand(-1, S0, -1, -1).contiguous().view(Bq, A, 6))
        tl = static["tl"]
        hist_tl = st["gt_tl"][:, :, tidx]                            # [n_sc, n_tl, S0, W, 5]
        hist_tl = (hist_tl.permute(0, 2, 1, 3, 4) * m8[None, :, None, :, None]).contiguous().view(Bq, n_tl, W, 5)
        rep = lambda x: x.repeat_interleave(S0, 0).contiguous()  # noqa: E731
        knn = lambda q: dict(idx=rep(q["idx"]), inv=rep(q["inv"]), rel=rep(q["rel"]))  # noqa: E731
        c0 = knn(tl["cross"][0])
        tlb = dict(n_sc=Bq, n_tl=n_tl, tl_token_invalid=rep(tl["tl_token_invalid"]),
                   tl_attr_rows=tl["tl_token_attr"].view(n_sc, 1, n_tl, 1, d).expand(-1, S0, -1, W, -1).reshape(-1, d).contiguous(),
                   knn_self=knn(tl["knn_self"]),
                   cross=[dict(c0, kv0=c["kv0"], T0=c["T0"], div0=S0, K0=c["K0"]) for c in tl["cross"]])
        a = torch.arange(A, device=dev, dtype=torch.int32)
        idx = [((s * A + a)[None, :].expand(st["B"], -1)).reshape(-1).contiguous() for s in range(S0)]
        return dict(stb=stb, tlb=tlb, hist_tl=hist_tl, d_rows=d_rows, idx=idx)

    def _warm_steps(self, st: dict, static: dict, navi: dict, n_steps: int) -> int:
        """Policy steps 1 .. S0: ONE batched pass of the TL and agent encoders over (scene, step) rows, then per step only
        the rollout-dependent part (heads with the rollout's latent / navigation, dynamics, bookkeeping). Leaves the TL
        pipeline primed for step S0 + 1. Returns the number of steps done."""
        m, lib, w = self.model, L.load(), self._warm
        S0, d, R = self._s0, m.d, self.R
        n_sc, A, n_tl = st["n_sc"], st["A"], st["n_tl"]
        tl_feat, logits = m.tl_forward(w["hist_tl"], w["d_rows"], w["tlb"])
        kv_tl = m.ag_tl_tables(tl_feat)
        x = m.ag_forward(w["stb"], static["mp"], static["kv_mp"], static["tl"], tl_feat, S0, kv_tl=kv_tl, tl_pose_div=S0)
        logits = logits.view(n_sc, S0, n_tl, -1).permute(1, 0, 2, 3).contiguous()                # [S0, n_sc * n_tl, 5]
        table = x.view(n_sc, S0 * A, d)
        n_do = min(S0, n_steps)
        for s in range(1, n_do + 1):
            ops.gather_rows(table, w["idx"][s - 1], A, R, out=st["x_cat"][:, :d])                # token of (scene, step) -> its R rollouts
            act = m.heads(st["x_cat"], st, navi)
            L.check(lib.tb_tl_step_ex(L.ptr(logits[s - 1]), L.ptr(ops._u8(static["tl"]["tl_token_invalid"])),
                                      L.ptr(st["gt_tl"]), st["n_gt"], L.ptr(st["d_step"]), st["Bt"], n_tl, m.W, self.T,
                                      L.ptr(st["hist_tl"]), L.ptr(st["tl_out"]), L.ptr(st.get("tl_nll")), L.stream()),
                    "tb_tl_step_ex")
            self._advance(st, static, act)
        # prime the software-pipelined TL branch: tokens of step n_do + 1 into its parity's buffer set
        st["d_step_tl"].fill_(n_do + 1)
        self._tl_branch(st, static, (n_do + 1) % 2)
        st["d_step_tl"].fill_(n_do + 2)
        self._host_step = n_do + 1
        return n_do

    # ---------------------------------------------------------------------------------------------- public API
    _AGENT_KEYS = {"sc/ag_valid": 1, "sc/ag_pose": 1, "sc/ag_motion": 1, "sc/ag_attr": 1, "ref/ag_type": 1, "ref/ag_size": 1,
                   "ag_latent": 2, "ag_latent_valid": 1, "ag_navi_valid": 1, "ref/ag_role": 1, "tf/forcing_agent": 1,
                   "player/valid": 2, "player/action": 2}  # player arrays are per rollout after _player_inputs

    def _player_inputs(self, batch: Dict[str, Tensor]) -> Dict[str, Tensor]:
        """Check the optional caller-control keys and bring the player arrays to the per-rollout layout:
        "player/valid" [n_sc, (R,) A] bool, "player/action" [n_sc, (R,) A, step_end, 2] (physical units: m/s^2, rad/s;
        step s reads column s-1), "tf/forcing_agent" [n_sc, A] bool. Raises ValueError on wrong shapes / dtypes and
        non-finite actions."""
        n_sc, A, _ = batch["sc/ag_valid"].shape
        R, T = self.R, self.T
        fa = batch.get("tf/forcing_agent")
        if fa is not None and (fa.dtype != torch.bool or tuple(fa.shape) != (n_sc, A)):
            raise ValueError(f"tf/forcing_agent: expected bool [{n_sc}, {A}], got {fa.dtype} {tuple(fa.shape)}")
        if "player/valid" not in batch:
            if "player/action" in batch:
                raise ValueError("player/action without player/valid")
            return batch
        pv, pa = batch["player/valid"], batch.get("player/action")
        if pv.dtype != torch.bool or tuple(pv.shape) not in ((n_sc, A), (n_sc, R, A)):
            raise ValueError(f"player/valid: expected bool [{n_sc}, ({R},) {A}], got {pv.dtype} {tuple(pv.shape)}")
        if pa is None:
            raise ValueError("player/valid needs player/action (begin() starts from a zero plan)")
        if not pa.is_floating_point() or tuple(pa.shape) not in ((n_sc, A, T, 2), (n_sc, R, A, T, 2)):
            raise ValueError(f"player/action: expected float [{n_sc}, ({R},) {A}, {T}, 2], got {pa.dtype} {tuple(pa.shape)}")
        if not bool(torch.isfinite(pa).all()):
            raise ValueError("player/action holds non-finite values")
        out = dict(batch)
        out["player/valid"] = pv if pv.dim() == 3 else pv[:, None].expand(-1, R, -1)
        out["player/action"] = (pa if pa.dim() == 5 else pa[:, None].expand(-1, R, -1, -1, -1)).float()
        return out

    def _compact(self, batch: Dict[str, Tensor]) -> Dict[str, Tensor]:
        """Drop the agent slots that are invalid at every ground-truth step in all scenes of the batch (see
        `compact_agents`). Returns the batch to load (the caller's dict is not modified)."""
        gt_valid = batch["sc/ag_valid"]
        n_sc, A, _ = gt_valid.shape
        self._perm, self._A_full = None, A
        if not self.compact_agents:
            return batch
        ever = gt_valid.any(-1)
        a_eff = max(int(ever.sum(1).max()), self.sz["k_ag2ag"] + 1)
        a_eff = min(A, (a_eff + 3) // 4 * 4)
        if a_eff >= A:
            return batch
        perm = torch.sort((~ever).to(torch.uint8), dim=1, stable=True)[1][:, :a_eff]           # valid first, original order kept
        out = dict(batch)

        def take(t, dim):
            idx = perm.to(t.device)
            shape = [1] * t.dim()
            shape[0], shape[dim] = n_sc, a_eff
            idx = idx.view(shape).expand([t.shape[i] if i != dim else a_eff for i in range(t.dim())])
            return torch.gather(t, dim, idx)

        for k, dim in self._AGENT_KEYS.items():
            if k in batch and batch[k].shape[0] == n_sc:
                out[k] = take(batch[k], dim)
        dest = batch["agent/dest"]
        out["agent/dest"] = take(dest, 1 if dest.dim() == 2 else 2)
        for k in ("ag_latent_valid", "ag_navi_valid"):  # [n_sc, A] or per rollout [n_sc * R, A]
            if k in batch and batch[k].shape[0] != n_sc:
                t = batch[k].view(n_sc, -1, A)
                out[k] = take(t, 2).reshape(-1, a_eff)
        self._perm = perm.to(self.dev)
        return out

    def prepare(self, batch: Dict[str, Tensor], static: Optional[dict] = None) -> dict:
        """Upload a batch of scenes, encode them (unless `static` is given) and build the step graph.
        Optional keys: "player/valid" + "player/action" (an open-loop plan for chosen agents, see `_player_inputs`)
        and "tf/forcing_agent" (log replay: these agents follow their ground truth wherever it is valid)."""
        batch = self._compact(self._player_inputs(batch))
        self._players, self._t = "player/valid" in batch, None
        n_sc, A, n_gt = batch["sc/ag_valid"].shape
        n_tl = batch["sc/tl_valid"].shape[1]
        _, n_mp, n_node = batch["sc/mp_valid"].shape
        shape = (n_sc, A, n_tl, n_gt, n_mp, n_node)
        self._sat.zero_()  # sticky from here on: scene encoding and every run() of this batch OR into it
        if self._shape != shape:
            # state buffers, scene tensors and step graphs are kept per shape (a few, LRU): with agent compaction
            # consecutive batches may differ in the number of agent slots, and a re-capture costs ~0.3 s
            if self._shape is not None:
                self._by_shape[self._shape] = (self._st, self._static, self._navi, self._graphs,
                                               getattr(self, "launches_per_step", 0))
                while len(self._by_shape) > 3:
                    self._by_shape.pop(next(iter(self._by_shape)))
            if shape in self._by_shape:
                self._st, self._static, self._navi, self._graphs, self.launches_per_step = self._by_shape.pop(shape)
            else:
                self._st, self._static, self._navi, self._graphs = self._alloc(*shape), None, None, {}
            self._shape = shape
        st = self._st
        self._load_state(st, batch)
        new_static = static if static is not None else self.encode_scenes(batch)
        new_navi = self.model.navi_static(new_static["mp"], st["dest_idx"], self.R)
        self.model.latent_static(new_navi, st)
        if self._graphs and _same_layout((self._static, self._navi), (new_static, new_navi)):
            # same shapes as the captured step graphs: refresh the scene tensors in place, keep the graphs
            _copy_tree((self._static, self._navi), (new_static, new_navi))
        else:
            self._static, self._navi, self._graphs = new_static, new_navi, {}
        self._s0 = self._invariant_steps(st) if (self.warm_dedup and self.tl_per_scene) else 0
        self._warm = self._build_warm(st, self._static) if self._s0 else None
        return st

    def run(self, n_steps: Optional[int] = None, record=None) -> Dict[str, Tensor]:
        """Run the closed loop from time 0 for n_steps (default: all). Returns views of the trajectory buffers."""
        st, n_steps = self._st, n_steps or self.T
        if not 1 <= n_steps <= self.T:  # pred_* / tl_out hold step_end columns; the kernels also refuse s > T
            raise ValueError(f"run(n_steps={n_steps}): the engine was built with step_end={self.T}")
        warm = self._s0 > 0 and record is None
        done = 0
        self._t = None
        if self.use_graph and record is None:
            graph = self._captured_graph()
            self._reset(st, tl_prologue=not warm)
            if warm:  # rollout-invariant warm-start steps: encoders once per scene, all steps in one batch
                done = self._warm_steps(st, self._static, self._navi, n_steps)
            self.graph_steps = n_steps - done
            for s_ in range(done + 1, n_steps + 1):
                graph[(s_ + 1) % 2].replay()
        else:
            self._reset(st, tl_prologue=not warm)
            if warm:
                done = self._warm_steps(st, self._static, self._navi, n_steps)
            self.graph_steps = 0
            for s_ in range(done + 1, n_steps + 1):
                aux = {} if record is not None else None
                n0 = ops.LAUNCHES
                self._step(st, self._static, self._navi, aux)
                self.launches_per_step = ops.LAUNCHES - n0
                if record is not None:
                    record(s_, aux)
        return self.results()

    def _captured_graph(self):
        """The (odd step, even step) graphs of the prepared batch's shape and player mode, captured on first use."""
        if self._graph is None:
            st = self._st
            self._reset(st)
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._step(st, self._static, self._navi)  # warm-up (allocator, lazy module load)
            torch.cuda.current_stream().wait_stream(s)
            self._reset(st)
            graphs = []
            for parity in (1, 0):  # first step is odd
                n0 = ops.LAUNCHES
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._step(st, self._static, self._navi, parity=parity)
                self.launches_per_step = ops.LAUNCHES - n0
                graphs.append(g)
            self._graphs[self._players] = (graphs[0], graphs[1])  # indexed by (step + 1) % 2: odd steps first
        return self._graph

    # ---------------------------------------------------------------------------------------------- step by step
    def begin(self, batch: Dict[str, Tensor], static: Optional[dict] = None) -> Dict[str, Tensor]:
        """Step-by-step stepping for closed-loop planners: `prepare` the batch, reset to time 0 and, when warm-start
        de-duplication applies, run its rollout-invariant steps 1 .. S0 (every valid agent is teacher-forced there, so a
        player only changes its own pred_* of those steps; they use the columns of batch["player/action"], a zero plan
        when the key is absent). Returns the observation at the current time t (see `step`)."""
        if "player/valid" in batch and "player/action" not in batch:
            n_sc, A, _ = batch["sc/ag_valid"].shape
            batch = dict(batch, **{"player/action": torch.zeros(n_sc, A, self.T, 2)})
        self.prepare(batch, static)
        st = self._st
        if self.use_graph:
            self._captured_graph()
        warm = self._s0 > 0
        self._reset(st, tl_prologue=not warm)
        self._t = self._warm_steps(st, self._static, self._navi, self.T) if warm else 0
        self.graph_steps = 0
        return self._observe()

    def step(self, player_action: Optional[Tensor] = None) -> Dict[str, Tensor]:
        """Policy step t + 1 of a rollout started with `begin`. `player_action` [n_sc, (R,) A, 2] (caller's agent order,
        physical units) becomes column t of the plan (a plain async copy), so the agents of batch["player/valid"]
        follow it in this step; None keeps the plan's column. Replays one step graph and returns the observation at
        the new time: dict(t=int, valid [n_sc*R, A] bool, pose / motion [n_sc*R, A, 3]) on the device. A fixed plan
        fed column by column gives the bits of `run()` with that plan."""
        t = self._t
        if t is None:
            raise RuntimeError("step() needs begin(batch) first")
        st = self._st
        if t >= self.T:
            raise RuntimeError(f"step(): the rollout reached step_end={self.T}")
        if player_action is not None:
            if not self._players:
                raise ValueError("step(player_action) needs a batch with player/valid")
            st["player_action"][:, :, t].copy_(self._plan_column(player_action), non_blocking=True)
        if self.use_graph:
            self._graph[t % 2].replay()  # step t + 1: odd steps use graph 0
        else:
            self._step(st, self._static, self._navi)
        self.graph_steps += 1
        self._t = t + 1
        return self._observe()

    def _plan_column(self, a: Tensor) -> Tensor:
        """[n_sc, (R,) A_caller, 2] actions -> [B, A, 2] on the device in the kept agent slots' order."""
        st, R = self._st, self.R
        n_sc, A = st["n_sc"], self._A_full
        if not a.is_floating_point() or tuple(a.shape) not in ((n_sc, A, 2), (n_sc, R, A, 2)):
            raise ValueError(f"player_action: expected float [{n_sc}, ({R},) {A}, 2], got {a.dtype} {tuple(a.shape)}")
        if not bool(torch.isfinite(a).all()):
            raise ValueError("player_action holds non-finite values")
        a = a.to(self.dev, torch.float32, non_blocking=True)
        a = a if a.dim() == 4 else a[:, None].expand(-1, R, -1, -1)
        if self._perm is not None:
            a = torch.gather(a, 2, self._perm[:, None, :, None].expand(-1, R, -1, 2))
        return a.reshape(st["B"], st["A"], 2)

    def _observe(self) -> Dict[str, Tensor]:
        st = self._st
        out = dict(valid=st["valid"].bool(), pose=st["pose"].clone(), motion=st["motion"].clone())
        if self._perm is not None:
            out = {k: self._caller_order(v) for k, v in out.items()}
        out["t"] = self._t
        return out

    def _caller_order(self, t: Tensor) -> Tensor:
        """[n_sc*R, A_kept, ...] -> [n_sc*R, A, ...] in the caller's agent order; dropped slots read as zeros."""
        n_sc, R, A = self._st["n_sc"], self.R, self._A_full
        sc = torch.arange(n_sc, device=self.dev)[:, None]
        full = t.new_zeros((n_sc, R, A) + tuple(t.shape[2:]))
        full[sc, :, self._perm] = t.view((n_sc, R, -1) + tuple(t.shape[2:])).transpose(1, 2)
        return full.view((n_sc * R, A) + tuple(t.shape[2:]))

    def results(self) -> Dict[str, Tensor]:
        st, R = self._st, self.R
        n_sc, A = st["n_sc"], st["A"]
        tl = st["tl_out"] if not self.tl_per_scene else st["tl_out"].repeat_interleave(R, 0)
        vio = {k: st[f"vio_{k}"].bool() for k in VIOLATIONS} if self.rule_checks else {}
        if self.record_feedback:
            vio.update(outside_map=st["fb_outside"].bool(), dest_reached=st["fb_reached"].bool())
        out = dict(**vio, pred_valid=st["pred_valid"].bool(), pred_pose=st["pred_pose"], pred_motion=st["pred_motion"],
                   final_valid=st["valid"].bool(), final_navi_valid=~st["navi_invalid"])
        if self._perm is not None:  # back to the caller's agent order; the dropped (never valid) slots read as zeros
            A = self._A_full
            out = {k: self._caller_order(v) for k, v in out.items()}
        out["tl_state"] = tl.bool()
        out["joint_pose"] = out["pred_pose"].view(n_sc, R, A, self.T, 3)
        return out

    @torch.no_grad()
    def post_process_wosac(self, res: Dict[str, Tensor], batch: Dict[str, Tensor], n_keep: int = 32,
                           step_future_start: Optional[int] = None, w_road_edge: float = 0.0,
                           use_wosac_col: bool = True) -> Dict[str, Tensor]:
        """The step right after the loop (WOSACPostProcessing._filter_futures + forward,
        wosac_post_processing.py:31-75; SURVEY 8(f) rank 4): keep the `n_keep` joint futures of every scene with the
        fewest role-weighted collision / road-edge violations (needs `rule_checks=True` when R > n_keep) and express
        them in the global frame (`scenario_center`, `scenario_yaw`). Only the kept futures leave the device
        (R = 128 -> 32 in the reference's submission config)."""
        R = self.R
        if R > n_keep and not self.rule_checks:
            raise RuntimeError("post_process_wosac with more than n_keep rollouts needs RolloutEngine(rule_checks=True)")
        n_sc = res["pred_pose"].shape[0] // R
        t0 = C.ROLLOUT_CFG["time_step_current"] if step_future_start is None else step_future_start
        g = lambda k: batch[k].to(self.dev)  # noqa: E731
        sel = score = None
        if R > n_keep:
            col = res["collided_wosac" if use_wosac_col else "collided"]
            score, sel = ops.future_filter(col, res["run_road_edge"], g("ref/ag_role").any(-1).contiguous(), n_sc, R, t0,
                                           w_road_edge, n_keep)
        pos, yaw = ops.traj_global(res["pred_pose"], sel, g("scenario_center"), g("scenario_yaw"), n_sc, R, t0)
        return dict(pos_sim=pos, yaw_sim=yaw, sel=sel, score=score)

    def post_process_womd(self, res: Dict[str, Tensor], batch: Dict[str, Tensor], scores: Optional[Tensor] = None,
                          k_pred: int = 6, use_ade: bool = True, mpa_nms_thresh=(2.0, 2.0, 2.0),
                          score_temperature: float = -1.0, step_future_start: Optional[int] = None
                          ) -> Dict[str, Tensor]:
        """WOMDPostProcessing.forward on the device (womd_post_processing.py:36-106 with the parameters of
        configs/model/sim_agent.yaml:170-177; SURVEY 8(f) rank 4): per agent, the k_pred most probable of the R joint
        futures, type-dependent ADE NMS of their scores, 2 Hz down-sampling. `scores` [n_sc, R, A] are the joint
        futures' log-probs (waymo_motion.py:632; None = uniform, as for reactive replay :610-613)."""
        R = self.R
        n_sc = res["pred_pose"].shape[0] // R
        t0 = C.ROLLOUT_CFG["time_step_current"] if step_future_start is None else step_future_start
        pose = res["pred_pose"]
        fut = pose.view(n_sc, R, *pose.shape[1:])[:, :, :, t0:].contiguous()
        n_fut = C.ROLLOUT_CFG["time_step_end"] - C.ROLLOUT_CFG["time_step_current"]  # track_future_samples
        trajs, sc, mode = ops.womd_post(fut, None if scores is None else scores.to(self.dev), batch["ref/ag_type"].to(self.dev),
                                        k_pred, use_ade, mpa_nms_thresh, score_temperature, 4, 5, n_fut)
        return dict(trajs=trajs, scores=sc, mode=mode)

    def check_fp16_range(self) -> None:
        """Raise if a 16-bit intermediate of the tensor-core mode saturated since the last reset (one 4-byte read,
        synchronises). The reference computes these in fp32; a checkpoint whose [q|u], [k|v] or ReLU hidden rows exceed
        65,504 must run with `precision=0`, or `model.kv_half = False` (tf32 projections, fp32 intermediates)."""
        if int(self._sat.item()) != 0:
            raise FloatingPointError("an fp16 intermediate of the tensor-core mode saturated at 65504: rerun this "
                                     "checkpoint with RolloutEngine(precision=0) or engine.model.kv_half = False")

    def rollout(self, batch: Dict[str, Tensor], n_steps: Optional[int] = None) -> Dict[str, Tensor]:
        self.prepare(batch)
        res = self.run(n_steps)
        if self.model.kv_half:
            self.check_fp16_range()
        return res
