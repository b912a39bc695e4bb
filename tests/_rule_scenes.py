"""Scenes for tb_rule_check (csrc/rule_check.cu) and their float64 replay through the oracle's RuleCheckOracle.

A scene holds the arrays in the layouts tb_rule_check takes: pred_valid / pred_pose / pred_motion [B, A, T(,3)],
ag_type [B, A, 3], ag_size [B/div, A, 3], the per-step traffic-light states [B/tl_div, n_tl, T, 5] (state of step s
at index s-1; the kernel reads it from slot s % W of the hist_tl ring), tl_valid / tl_pose [B/div, n_tl(,3)] and the
raw map (mp_valid / mp_type / mp_pos / mp_dir [B/div, n_mp, n_node(,..)]) that engine.rule_tables turns into the
kernel's tables.

Flags are compared exactly, so no input may sit on a knife edge. Every builder runs one jitter-stability filter
instead of per-check margins: the float64 oracle is evaluated on the scene and on copies with every pose moved by
+-1e-4 m and every yaw by +-1e-5 rad, and each agent whose flags (or passive counter) change at any step is redrawn.
A builder fails if an unstable agent remains after a bounded number of redraws.

Agents are drawn in "cases" (a case is a small group of agents, traffic lights and polylines that belong together);
a case is redrawn as a whole from its own seed, so a redraw does not move the rest of the scene.
"""
import functools
import math
from types import SimpleNamespace

import torch

from oracle import tb_oracle as O
from trafficbotsv1_5_b200.engine import rule_tables

VIO = ("collided", "collided_wosac", "run_road_edge", "run_red_light", "passive")
QCAP = 4096       # rule_check.cu QCAP: candidate queue of one rollout-scene (agent pairs, then (polyline, vehicle) pairs)
MAX_A = 256       # rule_check.cu MAX_A: agents per rollout-scene
SIZE_SCALE = 1.1  # TrafficRuleChecker's ag_size scale (collisions, road edge); red light uses the unscaled size
W = 11            # history ring length of the engine (slot s % W holds the TL state of step s)
VEH, PED, CYC = (True, False, False), (False, True, False), (False, False, True)
LANE_T, EDGE_T, OTHER_T = (0, 1, 2), (4, 5, 7), (3, 9)  # map types: lane centre, road edge, neither
RED = 1
JITTER_XY, JITTER_YAW = 1e-4, 1e-5
YAWS = (0.0, math.pi / 2, -math.pi / 2, math.pi, -math.pi, 7.0, -20.0)


# ------------------------------------------------------------------------------------------------ scene assembly
class _Row:
    """One rollout-scene under construction (used with div = tl_div = 1)."""

    def __init__(self, T):
        self.T, self.ag, self.tl, self.pl, self.expect = T, [], [], [], []

    def agent(self, case, xy, yaw, length, width, kind=VEH, speed=0.0, valid=True, vel=0.0):
        """Static pose (or moving at `vel` m/s along the heading); `speed` is the motion the checks read."""
        v = torch.full((self.T,), bool(valid)) if isinstance(valid, bool) else torch.as_tensor(valid, dtype=torch.bool)
        self.ag.append(dict(case=case, xy=(float(xy[0]), float(xy[1])), yaw=float(yaw), size=(length, width),
                            kind=kind, speed=speed, valid=v, vel=vel))
        return len(self.ag) - 1

    def light(self, xy, state, valid=True):
        st = torch.full((self.T,), int(state)) if isinstance(state, int) else torch.as_tensor(state)
        self.tl.append(dict(xy=(float(xy[0]), float(xy[1])), state=st, valid=valid))

    def poly(self, pts, typ, valid=None):
        """Polyline through the points: node k = pts[k], dir = pts[k+1] - pts[k] (the last node's segment is empty)."""
        pts = torch.as_tensor(pts, dtype=torch.float64)
        d = torch.zeros_like(pts)
        d[:-1] = pts[1:] - pts[:-1]
        v = torch.ones(len(pts), dtype=torch.bool) if valid is None else torch.as_tensor(valid, dtype=torch.bool)
        self.pl.append(dict(pos=pts, dir=d, valid=v, typ=typ))

    def want(self, a, flag, steps):
        """Expected pattern of one flag of agent a: a bool per step."""
        self.expect.append((a, flag, torch.as_tensor(steps, dtype=torch.bool)))


def _stack(rows, n_node):
    """Rows (div = tl_div = 1) -> scene; agents, lights and polylines padded with invalid entries."""
    B, T = len(rows), rows[0].T
    A = max(1, max(len(r.ag) for r in rows))
    n_tl = max(1, max(len(r.tl) for r in rows))
    n_mp = max(1, max(len(r.pl) for r in rows))
    s = SimpleNamespace(div=1, tl_div=1, T=T)
    s.pred_valid = torch.zeros(B, A, T, dtype=torch.bool)
    s.pred_pose, s.pred_motion = torch.zeros(B, A, T, 3), torch.zeros(B, A, T, 3)
    s.ag_type, s.ag_size = torch.zeros(B, A, 3, dtype=torch.bool), torch.zeros(B, A, 3)
    s.tl_state = torch.zeros(B, n_tl, T, 5, dtype=torch.bool)
    s.tl_state[..., 3] = True
    s.tl_valid, s.tl_pose = torch.zeros(B, n_tl, dtype=torch.bool), torch.zeros(B, n_tl, 3)
    s.mp_valid = torch.zeros(B, n_mp, n_node, dtype=torch.bool)
    s.mp_type = torch.zeros(B, n_mp, 11, dtype=torch.bool)
    s.mp_type[..., OTHER_T[1]] = True
    s.mp_pos, s.mp_dir = torch.zeros(B, n_mp, n_node, 2), torch.zeros(B, n_mp, n_node, 2)
    s.case = torch.full((B, A), -1, dtype=torch.long)
    s.expect = []
    t = torch.arange(T, dtype=torch.float64)
    for b, r in enumerate(rows):
        for a, g in enumerate(r.ag):
            hd = (math.cos(g["yaw"]), math.sin(g["yaw"]))
            s.pred_valid[b, a] = g["valid"]
            s.pred_pose[b, a, :, 0] = (g["xy"][0] + 0.1 * g["vel"] * t * hd[0]).float()
            s.pred_pose[b, a, :, 1] = (g["xy"][1] + 0.1 * g["vel"] * t * hd[1]).float()
            s.pred_pose[b, a, :, 2] = g["yaw"]
            s.pred_motion[b, a, :, 0] = g["speed"]
            s.ag_type[b, a] = torch.tensor(g["kind"])
            s.ag_size[b, a, 0], s.ag_size[b, a, 1], s.ag_size[b, a, 2] = g["size"][0], g["size"][1], 1.5
            s.case[b, a] = g["case"]
        for j, g in enumerate(r.tl):
            s.tl_state[b, j] = torch.nn.functional.one_hot(g["state"], 5).bool()
            s.tl_valid[b, j] = g["valid"]
            s.tl_pose[b, j, 0], s.tl_pose[b, j, 1] = g["xy"]
        for k, g in enumerate(r.pl):
            n = len(g["pos"])
            assert n <= n_node
            s.mp_pos[b, k, :n], s.mp_dir[b, k, :n], s.mp_valid[b, k, :n] = g["pos"].float(), g["dir"].float(), g["valid"]
            s.mp_type[b, k] = False
            s.mp_type[b, k, g["typ"]] = True
        s.expect += [(b, a, f, st) for a, f, st in r.expect]
    return s


def kernel_tables(s):
    """engine.rule_tables of the scene's map ([B/div, ...])."""
    return rule_tables(s.mp_valid, s.mp_type, s.mp_pos, s.mp_dir)


# ------------------------------------------------------------------------------------------------ the reference
def replay(s, dtype=torch.float64, pose_offset=None, with_counters=False):
    """RuleCheckOracle over steps 1..T on `dtype` copies of the scene's inputs, with the kernel's row mapping
    (scene row b // div, TL row b // tl_div). Returns {flag: [B, A, T] bool} and the final passive counter
    (and the counter after every step with `with_counters`)."""
    B, A, T = s.pred_valid.shape
    rows, trows = torch.arange(B) // s.div, torch.arange(B) // s.tl_div
    f = lambda t: t.to(dtype)  # noqa: E731
    oc = O.RuleCheckOracle(s.mp_valid[rows], s.mp_type[rows], f(s.mp_pos[rows]), f(s.mp_dir[rows]), s.ag_type,
                           f(s.ag_size[rows]), s.tl_valid[rows], f(s.tl_pose[rows]), size_scale=SIZE_SCALE)
    out = {k: [] for k in VIO}
    counters = []
    for t in range(T):
        pose = f(s.pred_pose[:, :, t])
        if pose_offset is not None:
            pose = pose + pose_offset
        for k, v in oc.check(s.pred_valid[:, :, t], pose, f(s.pred_motion[:, :, t]), s.tl_state[trows, :, t]).items():
            out[k].append(v)
        counters.append(oc.counter.clone())
    flags = {k: torch.stack(v, 2) for k, v in out.items()}
    if with_counters:
        return flags, oc.counter, torch.stack(counters, 2)
    return flags, oc.counter


def unstable(s, n_copies=4, seed=0):
    """[B, A] bool: agents whose float64 flags or passive counter change at any step when every pose is moved by
    +-JITTER_XY and every yaw by +-JITTER_YAW (independent signs per agent and coordinate, n_copies draws)."""
    base, _, cnt = replay(s, with_counters=True)
    g = torch.Generator().manual_seed(seed)
    B, A, _ = s.pred_valid.shape
    bad = torch.zeros(B, A, dtype=torch.bool)
    scale = torch.tensor([JITTER_XY, JITTER_XY, JITTER_YAW], dtype=torch.float64)
    for _ in range(n_copies):
        sign = torch.randint(0, 2, (B, A, 3), generator=g).to(torch.float64) * 2 - 1
        fl, _, c = replay(s, pose_offset=sign * scale, with_counters=True)
        for k in VIO:
            bad |= (fl[k] != base[k]).any(-1)
        bad |= (c != cnt).any(-1)
    return bad


def _stabilised(make, seed, rounds=12):
    """make(gen_of) -> scene, where gen_of(case) gives the generator of a case. Cases holding an unstable agent are
    redrawn from a new seed until none is left."""
    bump = {}

    def gen_of(case):
        return torch.Generator().manual_seed(seed * 1_000_003 + case * 7919 + bump.get(case, 0) * 104_729)

    for _ in range(rounds):
        s = make(gen_of)
        bad = unstable(s, seed=seed)
        if not bool(bad.any()):
            return s
        for case in set(s.case[bad].tolist()):
            assert case >= 0, "an unstable agent belongs to no case"
            bump[case] = bump.get(case, 0) + 1
    raise AssertionError(f"{int(bad.sum())} agents still on a knife edge after {rounds} redraws")


def _U(g, lo, hi):
    return float(torch.rand((), generator=g, dtype=torch.float64)) * (hi - lo) + lo


def _frame(xy, yaw):
    c, s = math.cos(yaw), math.sin(yaw)
    return lambda u, v: (xy[0] + u * c - v * s, xy[1] + u * s + v * c)  # noqa: E731


def _origin(k):
    """Case slots 30 m apart (beyond every interaction range of the checks), within +-60 m."""
    return ((k % 4) * 30.0 - 45.0, (k // 4) * 30.0 - 45.0)


def _size(kind, g):
    if kind == PED:
        w = _U(g, 0.6, 1.0)
        return w, w
    if kind == CYC:
        return _U(g, 1.6, 2.0), _U(g, 0.6, 0.8)
    return _U(g, 4.0, 5.0), _U(g, 1.8, 2.1)


def _rows(cases, T, per_row=16):
    """cases: list of fn(row, case_id, origin, gen). Returns make(gen_of) laying them out 16 to a row."""
    def make(gen_of, n_node):
        rows = []
        for k, fn in enumerate(cases):
            if k % per_row == 0:
                rows.append(_Row(T))
            fn(rows[-1], k, _origin(k % per_row), gen_of(k))
        return _stack(rows, n_node)
    return make


# ------------------------------------------------------------------------------------------------ hand-placed builders
def _pair_case(ta, tb, geom, overlap, yaw0):
    """Two agents at a controlled overlap (2-10 cm) or gap: side by side, nose to tail, corner to corner (aligned boxes,
    along the diagonal) or a corner of b (turned) into the flat side of a. Rounded (WOSAC) corners are recessed by more
    than 10 cm, so corner contacts give `collided` without `collided_wosac`; pedestrian pairs never give `collided`."""
    def fn(row, case, o, g):
        La, Wa = _size(ta, g)
        Lb, Wb = _size(tb, g)
        yaw = yaw0 + _U(g, -0.05, 0.05)
        eps = _U(g, 0.02, 0.10) * (1 if overlap else -1)
        k = SIZE_SCALE
        to = _frame(o, yaw)
        rel = 0.0
        if geom == "side":
            u, v = _U(g, -0.3, 0.3), (Wa + Wb) / 2 * k - eps
        elif geom == "nose":
            u, v = (La + Lb) / 2 * k - eps, _U(g, -0.2, 0.2)
        elif geom == "corner":
            du, dv = (La + Lb) / 2 * k, (Wa + Wb) / 2 * k
            n = math.hypot(du, dv)
            u, v = du - eps * du / n, dv - eps * dv / n
        else:  # "corner_side": b turned so that one corner points at a's side
            beta = math.atan2(Wb, Lb)
            rel = -math.pi / 2 - beta
            u, v = _U(g, -0.3, 0.3), Wa / 2 * k + math.hypot(Lb, Wb) / 2 * k - eps
        a = row.agent(case, to(0.0, 0.0), yaw, La, Wa, ta)
        b = row.agent(case, to(u, v), yaw + rel, Lb, Wb, tb)
        both_ped = ta == PED and tb == PED
        col = overlap and not both_ped
        wosac = overlap and geom in ("side", "nose")
        for i in (a, b):
            row.want(i, "collided", [col] * row.T)
            row.want(i, "collided_wosac", [wosac] * row.T)
    return fn


def _invalid_overlap(row, case, o, g):
    """An invalid agent overlapping a valid one (and a valid pedestrian far enough away): no flag on either."""
    yaw = _U(g, -math.pi, math.pi)
    to = _frame(o, yaw)
    a = row.agent(case, to(0, 0), yaw, 4.5, 2.0, VEH)
    b = row.agent(case, to(1.0, 0.4), yaw + 0.3, 4.5, 2.0, VEH, valid=False)
    c = row.agent(case, to(0.5, -0.2), yaw, 0.8, 0.8, PED, valid=False)
    for i in (a, b, c):
        row.want(i, "collided", [False] * row.T)
        row.want(i, "collided_wosac", [False] * row.T)


@functools.lru_cache(maxsize=None)
def pairs():
    cases = []
    i = 0
    for ta, tb in ((VEH, VEH), (VEH, PED), (PED, PED)):
        for geom in ("side", "nose", "corner", "corner_side"):
            for overlap in (True, False):
                cases.append(_pair_case(ta, tb, geom, overlap, YAWS[i % len(YAWS)]))
                i += 1
    cases.append(_invalid_overlap)
    make = _rows(cases, T=2)
    return _stabilised(lambda gen_of: make(gen_of, 4), seed=11)


def _edge_case(what):
    """A vehicle (or another agent type) and one polyline placed in the agent's frame against its scaled box."""
    def fn(row, case, o, g):
        kind = {"ped": PED, "cyc": CYC}.get(what, VEH)
        L, Wd = _size(kind, g)
        yaw = _U(g, -4.0, 4.0)
        to = _frame(o, yaw)
        a = row.agent(case, to(0, 0), yaw, L, Wd, kind)
        lh, wh = L / 2 * SIZE_SCALE, Wd / 2 * SIZE_SCALE
        u = _U(g, -0.8, 0.8) * min(lh, 1.0)
        typ = EDGE_T[case % 3]
        cross = [to(u, wh + _U(g, 0.2, 0.6)), to(u + _U(g, -0.2, 0.2), wh - _U(g, 0.2, 0.5))]
        hit = False
        if what == "cross":
            row.poly(cross, typ)
            hit = True
        elif what == "front":
            v = _U(g, -0.5, 0.5) * wh
            row.poly([to(lh - _U(g, 0.2, 0.5), v), to(lh + _U(g, 0.2, 0.5), v + 0.1)], typ)
            hit = True
        elif what == "late_node":  # 7 nodes, the box edge lies between nodes 4 and 5
            y0 = wh + 2.6 - _U(g, 0.02, 0.1)
            row.poly([to(u, y0 - 0.5 * n) for n in range(7)], typ)
            hit = True
        elif what == "inside":
            row.poly([to(-0.5 * lh, -0.3 * wh), to(0.6 * lh, 0.4 * wh)], typ)
        elif what == "outside_5cm":
            row.poly([to(-0.8 * lh, wh + 0.05), to(0.8 * lh, wh + 0.05)], typ)
            row.poly([to(u, wh + 1.0), to(u, wh + 0.05)], typ)
        elif what == "invalid_node":
            row.poly(cross, typ, valid=[False, True])
        elif what == "all_invalid":
            row.poly(cross, typ, valid=[False, False])
        elif what == "lane":
            row.poly(cross, LANE_T[case % 3])
        else:  # a pedestrian / cyclist crossing an edge
            row.poly(cross, typ)
        row.want(a, "run_road_edge", [hit] * row.T)
    return fn


@functools.lru_cache(maxsize=None)
def road_edge():
    whats = ("cross", "front", "late_node", "inside", "outside_5cm", "invalid_node", "all_invalid", "lane", "ped", "cyc")
    cases = [_edge_case(w) for w in whats for _ in range(2)]
    make = _rows(cases, T=2)
    return _stabilised(lambda gen_of: make(gen_of, 7), seed=12)


def _red_case(what):
    """A vehicle with speed v and one traffic light placed in its frame against the red-light rectangle, half-extents
    0.3 * length along and 0.9 * width across (UNscaled size), now and after the 0.1 s step."""
    def fn(row, case, o, g):
        kind = PED if what == "ped" else VEH
        L, Wd = (4.5, 2.0) if kind == VEH else (0.8, 0.8)
        L, Wd = L + _U(g, -0.3, 0.3), Wd + _U(g, -0.1, 0.1)
        yaw = _U(g, -7.0, 7.0)
        to = _frame(o, yaw)
        ln, wd = 0.3 * L, 0.9 * Wd
        band = 0.03 * L  # scaled - unscaled half-extent along
        d = _U(g, 0.03, 0.1)
        ty = _U(g, -0.6, 0.6) * wd
        state, valid, hit = RED, True, True
        if what == "stay":
            tx, step, hit = -ln + 1.0, 0.5, False
        elif what == "band_now":      # in the band now: only a kernel using the scaled size sees it inside
            tx, step, hit = -ln - 0.5 * band, 0.5, False
        elif what == "band_after":    # inside now, in the band after: a kernel using the scaled size misses it
            tx, step = -ln + d, d + 0.5 * band
        elif what == "band_side":     # in the band across the heading
            tx, ty, step, hit = -ln + 0.3, (0.9 + 0.045) * Wd, 0.6, False
        else:
            tx, step = -ln + d, d + _U(g, 0.3, 0.6)
        if what == "not_red":
            state, hit = (0, 2, 3, 4)[case % 4], False
        elif what == "invalid":
            valid, hit = False, False
        elif what == "ped":
            hit = False
        steps = [hit] * row.T
        if what == "switching":       # red on odd steps, state 3 on even steps
            state = torch.tensor([RED if (s + 1) % 2 else 3 for s in range(row.T)])
            steps = [bool((s + 1) % 2) for s in range(row.T)]
        a = row.agent(case, to(0, 0), yaw, L, Wd, kind, speed=step / 0.1)
        row.light(to(tx, ty), state, valid)
        row.want(a, "run_red_light", steps)
    return fn


@functools.lru_cache(maxsize=None)
def red_light():
    whats = ("leave", "stay", "band_now", "band_after", "band_side", "not_red", "invalid", "ped", "switching")
    cases = [_red_case(w) for w in whats for _ in range(2)] + [_red_case("not_red") for _ in range(2)]
    make = _rows(cases, T=14)
    return _stabilised(lambda gen_of: make(gen_of, 4), seed=13)


PASSIVE_T = 30


def _passive_case(what):
    """A slow vehicle beside a lane-centre polyline (nodes 1 m apart along its heading), with the things that block the
    passive check placed around it. `first` is the step at which the flag first appears (None: never)."""
    def fn(row, case, o, g):
        yaw = _U(g, -3.2, 3.2)
        to = _frame(o, yaw)
        L, Wd = 4.5 + _U(g, -0.3, 0.3), 1.9
        speed, lat, first = _U(g, 0.5, 4.0), 1.9, 21
        if what == "lane_2.1":
            lat, first = 2.1, None
        elif what == "speed_4.9":
            speed = 4.9
        elif what == "speed_5.1":
            speed, first = 5.1, None
        if what == "end_node":  # small vehicle 1.9 m past the end node of a lane, outside its bounding circle
            L, Wd = 3.0, 1.6
            row.poly([to(-1.9 - (19 - k), 0.0) for k in range(20)], LANE_T[case % 3])
        else:
            row.poly([to(-10.0 + k, lat) for k in range(20)], LANE_T[case % 3])
        a = row.agent(case, to(0, 0), yaw, L, Wd, VEH, speed=speed)
        if what.startswith("tl_"):
            _, dist, ang, state = what.split("_")
            dist, ang, state = float(dist), math.radians(float(ang)), int(state)
            row.light(to(dist * math.cos(ang), dist * math.sin(ang) * (1 if case % 2 else -1)), state)
            blocks = state != 3 and dist < 10 and math.cos(ang) > 0.95
            first = None if blocks else 21
        if what == "agent_ahead":  # a pedestrian 5 m ahead at steps 6 and 7: the counter resets and restarts at 8
            row.agent(case, to(5.0, 0.3), yaw, 0.8, 0.8, PED, valid=[s in (5, 6) for s in range(row.T)])
            first = 8 + 20
        row.want(a, "passive", [first is not None and s + 1 >= first for s in range(row.T)])
    return fn


@functools.lru_cache(maxsize=None)
def passive():
    whats = ["lane_1.9", "lane_2.1", "speed_4.9", "speed_5.1", "agent_ahead", "end_node"]
    whats += [f"tl_9.5_17_{st}" for st in range(5)] + ["tl_10.5_10_1", "tl_9.5_19.5_1", "tl_9.5_19.5_0"]
    make = _rows([_passive_case(w) for w in whats], T=PASSIVE_T)
    return _stabilised(lambda gen_of: make(gen_of, 20), seed=14)


@functools.lru_cache(maxsize=None)
def single_agent():
    """A = 1: a road-edge crossing, a red-light runner and a passive vehicle, one per rollout-scene."""
    cases = [_edge_case("cross"), _red_case("leave"), _passive_case("lane_1.9")]

    def make(gen_of):
        rows = []
        for k, fn in enumerate(cases):
            rows.append(_Row(22))
            fn(rows[-1], k, (0.0, 0.0), gen_of(k))
        return _stack(rows, 20)
    return _stabilised(make, seed=15)


# ------------------------------------------------------------------------------------------------ queue overflows
def pair_queue_count(s):
    """[B] ordered agent pairs the kernel queues: both valid, circumcircles of the SCALED size (+1e-3) touching."""
    B, A, _ = s.pred_valid.shape
    sz = s.ag_size[torch.arange(B) // s.div].double()[..., :2] * SIZE_SCALE
    rad = 0.5 * sz.norm(dim=-1) + 1e-3
    out = torch.zeros(B, s.T, dtype=torch.long)
    for t in range(s.T):
        v, xy = s.pred_valid[:, :, t], s.pred_pose[:, :, t, :2].double()
        d2 = ((xy[:, :, None] - xy[:, None]) ** 2).sum(-1)
        m = v[:, :, None] & v[:, None] & ~torch.eye(A, dtype=torch.bool) & (d2 <= (rad[:, :, None] + rad[:, None]) ** 2)
        out[:, t] = m.sum((1, 2))
    return out


def map_queue_count(s):
    """[B, T] (polyline, vehicle) pairs the kernel queues: polylines with a kind bit, valid vehicles, the rule_tables
    bounding circle within the map reach max(scaled circumradius + 1e-3, 2.001) of the vehicle."""
    B = s.pred_valid.shape[0]
    rows = torch.arange(B) // s.div
    tab = kernel_tables(s)
    circ, kind = tab["poly_circle"][rows].double(), tab["poly_kind"][rows]
    sz = s.ag_size[rows].double()[..., :2] * SIZE_SCALE
    reach = (0.5 * sz.norm(dim=-1) + 1e-3).clamp(min=2.001)
    out = torch.zeros(B, s.T, dtype=torch.long)
    for t in range(s.T):
        vv = s.pred_valid[:, :, t] & s.ag_type[:, :, 0]
        xy = s.pred_pose[:, :, t, :2].double()
        d2 = ((circ[:, :, None, :2] - xy[:, None]) ** 2).sum(-1)
        m = (kind[:, :, None] > 0) & vv[:, None] & (d2 <= (circ[:, :, None, 2] + reach[:, None]) ** 2)
        out[:, t] = m.sum((1, 2))
    return out


@functools.lru_cache(maxsize=None)
def crowd():
    """A = 256 long vehicles (16-22 m, 1.3-1.5 m wide) in 32 parallel lanes 1.95 m apart, 8 per lane at 22 m spacing:
    circumcircles reach ~18 neighbours (more than 4096 queued pairs), while boxes touch only nose to tail or, for the
    few slightly turned vehicles, at a corner."""
    T = 2

    def make(gen_of):
        row = _Row(T)
        for i in range(MAX_A):
            g = gen_of(i)
            lane, slot = i // 8, i % 8
            L, Wd = _U(g, 16.0, 22.0), _U(g, 1.3, 1.5)
            yaw = _U(g, -0.01, 0.01) + (math.pi if lane % 5 == 2 else 0.0) + (_U(g, -0.05, 0.05) if i % 9 == 4 else 0.0)
            xy = ((slot - 3.5) * 22.0 + _U(g, -0.5, 0.5), (lane - 15.5) * 1.95 + _U(g, -0.1, 0.1))
            row.agent(i, xy, yaw, L, Wd, VEH, speed=_U(g, 0, 8), valid=i % 61 != 7, vel=_U(g, 0.0, 3.0))
        row.light((0.0, 0.0), 3, valid=False)
        return _stack([row], 4)
    return _stabilised(make, seed=16, rounds=20)


@functools.lru_cache(maxsize=None)
def dense_map():
    """128 vehicles among 1100 short polylines (4 nodes, 2 m apart) in a 44 m square: more than 4096 queued (polyline,
    vehicle) pairs; 85 % of the polylines are lanes, 4 % road edges, the rest of no checked type."""
    T, n_pl, A = 2, 1100, 128

    def make(gen_of):
        g = torch.Generator().manual_seed(4242)
        row = _Row(T)
        for k in range(n_pl):
            x0, y0, h = _U(g, -22.0, 22.0), _U(g, -22.0, 22.0), _U(g, -math.pi, math.pi)
            r = float(torch.rand((), generator=g))
            typ = LANE_T[k % 3] if r < 0.85 else (EDGE_T[k % 3] if r < 0.89 else OTHER_T[k % 2])
            valid = [n != 2 for n in range(4)] if k % 17 == 3 else None
            row.poly([(x0 + 2.0 * n * math.cos(h), y0 + 2.0 * n * math.sin(h)) for n in range(4)], typ, valid)
        for i in range(A):
            ga = gen_of(i)
            L, Wd = _U(ga, 3.0, 5.0), _U(ga, 1.6, 2.1)
            kind = CYC if i % 19 == 4 else VEH
            row.agent(i, (_U(ga, -22.0, 22.0), _U(ga, -22.0, 22.0)), _U(ga, -math.pi, math.pi), L, Wd, kind,
                      speed=_U(ga, 0.0, 8.0), vel=_U(ga, 0.0, 2.0))
        row.light((0.0, 0.0), 3, valid=False)
        return _stack([row], 4)
    return _stabilised(make, seed=17, rounds=20)


# ------------------------------------------------------------------------------------------------ engine layout
@functools.lru_cache(maxsize=None)
def mixed(n_sc=2, R=3, tl_per_rollout=False, T=26, A=24):
    """Rollout-scene b uses map / TL / agent-size row b // R (div = R). TL states are per scene (tl_div = R, the
    engine's layout) or per rollout (tl_div = 1). Scenes differ in map, TLs, TL states and agent sizes; rollouts
    differ in agent poses, so a wrong row index changes flags. Agents move (0.1 s steps) and are placed around the
    scene's traffic lights, lane centres and road edges. T > W: the history ring wraps."""
    B, n_tl, n_lane, n_edge, n_node = n_sc * R, 6, 6, 6, 20
    Bt = B if tl_per_rollout else n_sc
    s = SimpleNamespace(div=R, tl_div=1 if tl_per_rollout else R, T=T)
    g = torch.Generator().manual_seed(900 + n_sc * 10 + R + (5 if tl_per_rollout else 0))
    U = lambda lo, hi: _U(g, lo, hi)  # noqa: E731
    s.tl_valid = torch.rand(n_sc, n_tl, generator=g) < 0.85
    s.tl_pose = torch.zeros(n_sc, n_tl, 3)
    s.tl_pose[..., :2] = torch.rand(n_sc, n_tl, 2, generator=g) * 60 - 30
    s.tl_state = torch.zeros(Bt, n_tl, T, 5, dtype=torch.bool)
    for r in range(Bt):
        for j in range(n_tl):
            st = []
            while len(st) < T:
                k = RED if float(torch.rand((), generator=g)) < 0.45 else int(torch.randint(0, 5, (), generator=g))
                st += [k] * int(torch.randint(2, 7, (), generator=g))
            s.tl_state[r, j] = torch.nn.functional.one_hot(torch.tensor(st[:T]), 5).bool()
    s.mp_valid = torch.ones(n_sc, n_lane + n_edge, n_node, dtype=torch.bool)
    s.mp_type = torch.zeros(n_sc, n_lane + n_edge, 11, dtype=torch.bool)
    s.mp_pos, s.mp_dir = torch.zeros(n_sc, n_lane + n_edge, n_node, 2), torch.zeros(n_sc, n_lane + n_edge, n_node, 2)
    lanes = []
    for sc in range(n_sc):
        for k in range(n_lane + n_edge):
            x0, y0, h = U(-30, 30), U(-30, 30), U(-math.pi, math.pi)
            step = 1.0 if k < n_lane else 0.6
            t = torch.arange(n_node, dtype=torch.float64)
            pos = torch.stack([x0 + step * t * math.cos(h), y0 + step * t * math.sin(h)], -1)
            s.mp_pos[sc, k] = pos.float()
            s.mp_dir[sc, k, :-1] = (pos[1:] - pos[:-1]).float()
            s.mp_type[sc, k, (LANE_T if k < n_lane else EDGE_T)[k % 3]] = True
            if k == n_lane + 1:
                s.mp_valid[sc, k, 7:] = False
            if k < n_lane:
                lanes.append((sc, x0, y0, h))
    kinds = [VEH if i % 10 < 8 else (PED if i % 10 == 8 else CYC) for i in range(A)]
    s.ag_type = torch.tensor([kinds] * B)
    s.ag_size = torch.zeros(n_sc, A, 3)
    for sc in range(n_sc):
        for i in range(A):
            L, Wd = _size(kinds[i], g)
            s.ag_size[sc, i, 0], s.ag_size[sc, i, 1], s.ag_size[sc, i, 2] = L, Wd, 1.5

    def make(gen_of):
        s.pred_valid = torch.zeros(B, A, T, dtype=torch.bool)
        s.pred_pose, s.pred_motion = torch.zeros(B, A, T, 3), torch.zeros(B, A, T, 3)
        s.case = torch.full((B, A), -1, dtype=torch.long)
        tt = torch.arange(T, dtype=torch.float64)
        for b in range(B):
            sc = b // R
            sl = [x for x in lanes if x[0] == sc]
            for i in range(A):
                ga = gen_of(b * A + i)
                L, Wd = float(s.ag_size[sc, i, 0]), float(s.ag_size[sc, i, 1])
                anchor = (i + b) % 3
                if anchor == 0:    # a traffic light ahead, inside or near the red-light rectangle
                    j = (i + b) % n_tl
                    yaw = _U(ga, -math.pi, math.pi)
                    tx, ty = float(s.tl_pose[sc, j, 0]), float(s.tl_pose[sc, j, 1])
                    u, v = _U(ga, -0.1, 0.9) * 0.3 * L, _U(ga, -1.0, 1.0) * 0.9 * Wd
                    c, sn = math.cos(yaw), math.sin(yaw)
                    x, y = tx - (u * c - v * sn), ty - (u * sn + v * c)
                    speed = _U(ga, 2.0, 12.0)
                elif anchor == 1:  # beside a lane centre, slow, along the lane
                    _, x0, y0, h = sl[(i + b) % len(sl)]
                    k, lat = _U(ga, 0, 19), _U(ga, -3.0, 3.0)
                    x, y = x0 + k * math.cos(h) - lat * math.sin(h), y0 + k * math.sin(h) + lat * math.cos(h)
                    yaw, speed = h + _U(ga, -0.2, 0.2), _U(ga, 0.0, 1.0) * (6.0 if i % 4 else 1.0)
                else:              # anywhere in the scene
                    x, y, yaw, speed = _U(ga, -30, 30), _U(ga, -30, 30), _U(ga, -math.pi, math.pi), _U(ga, 0, 10)
                vel = speed if i % 2 else 0.0
                s.pred_pose[b, i, :, 0] = (x + 0.1 * vel * tt * math.cos(yaw)).float()
                s.pred_pose[b, i, :, 1] = (y + 0.1 * vel * tt * math.sin(yaw)).float()
                s.pred_pose[b, i, :, 2] = yaw
                s.pred_motion[b, i, :, 0] = speed
                v = torch.ones(T, dtype=torch.bool)
                if i % 7 == 3:
                    v[int(_U(ga, 0, T - 4)):][:3] = False
                s.pred_valid[b, i] = v
                s.case[b, i] = b * A + i
        return SimpleNamespace(**vars(s))
    return _stabilised(make, seed=18 + (1 if tl_per_rollout else 0), rounds=16)


BUILDERS = dict(pairs=pairs, road_edge=road_edge, red_light=red_light, passive=passive, single_agent=single_agent,
                crowd=crowd, dense_map=dense_map, mixed_per_scene=lambda: mixed(), mixed_per_rollout=lambda: mixed(tl_per_rollout=True))
