"""The tensor-core tile kernels (csrc/tile_kernels.cu, tile_tc_device.cuh) against the oracle at the tile shapes that
only appear when a CTA holds several envs: balanced CTAs of 9-10 envs (the benchmark's 4 096 envs), the four-CTA
(DENSE) build, ragged last CTAs, every envs-per-CTA count of the run-time-N path including 128 mod N != 0, and one env
per CTA with 116 inactive threads.  ``tile_grid_plan`` spreads B <= 3 x 148 envs one per CTA, so the other parity
tests (B <= 200) never run these shapes.

1. Per-tick oracle along the kernel's own trajectory.  The generic rollout traces state, actions, Q, rewards and
   flags; tick t is judged on the kernel's own input state S_t, so the comparison never depends on trajectories
   staying together:
     * Q against a float64 evaluation of the reference network on the graph the oracle builds from S_t, per agent row
       relative to max |Q64| of the row, <= Q_BOUND (the float32 oracle's error on the same rows is printed);
     * the traced action is the first-index argmax of the traced Q, and the argmax of Q64 except where Q64's top-2
       gap is <= 2 Q_BOUND |Q64|max (counted and bounded);
     * the world step of the oracle from (S_t, action) reproduces state, flags and rewards: bit-exact where no contact
       force acts, 1e-6 relative under contact (GoTo rewards judged per env), flags exact;
     * returns are the tick-ordered sum of the traced rewards, hits the number of HIT flags.
2. The PLAIN instantiation (greedy complete-graph rollout, nothing traced) one tick at a time from states of a generic
   rollout, against the float32 oracle's greedy step; envs with an agent whose Q64 top-2 gap lies inside the band are
   skipped (their share is bounded).  Non-zero returns / hits go in and must be added to.
3. Stretched logits: conv1.att_src / att_dst scaled so that the in-env logit spread exceeds 100.  The softmax is then
   nearly one-hot and its shift (the maximum) decides whether the exponentials overflow.

Bounds.  Worst per-row error relative to max |Q64| over all ticks of a case, measured on one B200 (1 000 W), kernel /
float32 oracle on the same rows:
    N = 12 complete OA   B 700 4.1e-7 / 3.4e-7   B 4 096 5.1e-7 / 5.3e-7   B 5 000 3.0e-7 / 2.7e-7
                         B 6 007 5.1e-7 / 5.5e-7
    N = 12 complete GoTo B 5 000 8.0e-7 / 5.0e-7
    N = 12 kNN k = 5     B 4 096 5.0e-7 / 3.7e-7       N = 12 radius 0.35   B 4 096 7.9e-7 / 4.8e-7
    run-time N           N 2 5.5e-7 / 3.8e-7   N 3 5.0e-7 / 3.7e-7   N 5 5.6e-7 / 3.6e-7   N 7 4.3e-7 / 4.8e-7
                         N 9 5.0e-7 / 3.8e-7   N 16 5.6e-7 / 4.7e-7  N 33 4.1e-7 / 5.3e-7  N 43 4.2e-7 / 5.3e-7
                         N 64 5.6e-7 / 1.0e-6  N 100 8.7e-7 / 4.6e-7 N 128 6.7e-7 / 4.6e-7
    forward              N 12 4.1e-7 / 3.2e-7  N 7 4.3e-7 / 3.4e-7   N 33 4.1e-7 / 3.5e-7
    stretched (x15)      rollout N 12 6.4e-6 / 6.9e-6   rollout N 7 1.0e-6 / 1.9e-6   forward N 33 5.1e-6 / 8.7e-6
Q_BOUND = 3e-6 for the shipped weights (3.5x the worst, 8.7e-7).  With stretched logits the float32 rounding of
logits of several hundred is what remains, for the oracle as for the kernel: Q_BOUND_STRETCHED = 1e-5, the project's
bar (1.6x the worst, 6.4e-6).  Excused argmax flips per case: at most 13 of 393 216 agent rows.  PLAIN step: at most
1 % of the envs skipped (GoTo; ObstacleAvoidance none).  The whole file takes about 5.5 minutes on a 16-core host,
almost all of it oracle time.
"""
import os

import pytest
import torch

from helpers import load_params

pytestmark = pytest.mark.gpu

Q_BOUND = 3e-6               # shipped weights
Q_BOUND_STRETCHED = 1e-5     # part 3 (the float32 oracle's own error is of the same size there)
STATE_RTOL = 1e-6
FLIP_SHARE = 2e-3            # excused argmax flips (Q64 top-2 gap inside the band), share of agent rows
SKIP_SHARE = 0.05            # PLAIN step: share of envs skipped for an in-band agent
EDGE_ROWS = 1 << 20          # oracle chunk: ~1 M edges (the float64 message tensor is 256 MB)
STRETCH = 15.0               # att_src / att_dst scale of part 3


def _sb():
    import swarm_b200
    return swarm_b200


def _dev():
    return torch.device("cuda:0")


def _scen(scenario):
    L = _sb()._lib
    return L.SCENARIO_GOTO if scenario == "go_to" else L.SCENARIO_OBSTACLE_AVOIDANCE


def _exp(scenario):
    return "GoTo" if scenario == "go_to" else "ObstacleAvoidance"


def _gmode(graph):
    L = _sb()._lib
    return {"complete": L.GRAPH_COMPLETE, "knn": L.GRAPH_KNN, "radius": L.GRAPH_RADIUS}[graph]


def _graph_arg(graph):
    return {"complete": 0, "knn": 5, "radius": 0.35}[graph]


def _stretched(params, scale=STRETCH):
    p = {k: v.clone() for k, v in params.items()}
    p["conv1.att_src"] *= scale
    p["conv1.att_dst"] *= scale
    return p


def _random_states(scenario, B, N, seed):
    """Squeezed, jittered grids (a third of the ObstacleAvoidance swarms on the obstacle) with random velocities, so
    that agent-agent and agent-obstacle contacts occur."""
    from oracle import swarm_oracle as so, batched_oracle as bo
    g = torch.Generator().manual_seed(seed)
    centers = torch.stack([so.draw_center(scenario, True, g) for _ in range(B)])
    if scenario == so.OBSTACLE_AVOIDANCE:
        centers[::3] = torch.tensor(list(so.OBSTACLE_POS)) + 0.1 * torch.randn(len(centers[::3]), 2, generator=g)
    pos, _ = bo.reset_grid(scenario, centers, N)
    scale = torch.rand(B, 1, 1, generator=g) * 0.6 + 0.4
    ctr = pos.mean(dim=1, keepdim=True)
    pos = ctr + (pos - ctr) * scale + 0.01 * torch.randn(B, N, 2, generator=g)
    vel = 0.3 * torch.randn(B, N, 2, generator=g)
    return torch.cat([pos, vel], dim=2).contiguous()


class _threads:
    """The float64 / float32 network evaluations only feed tolerance checks: let them use the host's cores (the suite
    runs single-threaded so that the bit-exact oracle world step never changes its reduction order)."""

    def __enter__(self):
        self.n = torch.get_num_threads()
        torch.set_num_threads(max(1, min(16, os.cpu_count() or 1)))

    def __exit__(self, *exc):
        torch.set_num_threads(self.n)


def _oracle_q(params, state, graph):
    """Q of the reference network on the oracle's graph of ``state`` (f32[B,N,4], CPU), in float64 and float32."""
    from oracle import swarm_oracle as so, batched_oracle as bo
    B, N, _ = state.shape
    p64 = {k: v.double() for k, v in params.items()}
    per_env = N * N + 1 if graph != "knn" else 2 * 5 * N + 1
    chunk = max(1, EDGE_ROWS // per_env)
    q64, q32 = [], []
    for b0 in range(0, B, chunk):
        st = state[b0:b0 + chunk]
        pos, vel = st[..., :2].contiguous(), st[..., 2:].contiguous()
        ei = bo.batch_edge_index(bo.graph_edges(pos, graph, _graph_arg(graph)), N)
        x = bo.node_features(pos, vel).reshape(-1, 7)
        with torch.no_grad(), _threads():
            q64.append(so.gatq_forward(p64, x.double(), ei).reshape(-1, N, 9))
            q32.append(so.gatq_forward(params, x, ei).reshape(-1, N, 9))
    return torch.cat(q64), torch.cat(q32)


def _q_errors(q, q64):
    """per agent row: max |q - q64| / max |q64|."""
    scale = q64.abs().amax(dim=-1, keepdim=True)
    return ((q.double() - q64).abs() / scale).amax(dim=-1)


def _in_band(q64, bound):
    """agent rows whose Q64 top-2 gap is inside the tolerance band (the float32 argmax may legitimately differ)."""
    top2 = torch.topk(q64, 2, dim=-1).values
    return (top2[..., 0] - top2[..., 1]) <= 2 * bound * q64.abs().amax(dim=-1)


def _check_q(label, q, q64, q32, act=None, bound=Q_BOUND):
    """Q within ``bound`` of float64; actions = first-index argmax of q, and = argmax Q64 outside the band.
    Returns (kernel error, float32-oracle error, excused flips)."""
    assert torch.isfinite(q).all(), f"{label}: non-finite Q"
    err = _q_errors(q, q64).max().item()
    err32 = _q_errors(q32, q64).max().item()
    assert err <= bound, f"{label}: Q error {err:.3e} vs float64 (float32 oracle {err32:.3e})"
    flips = 0
    if act is not None:
        assert torch.equal(act.long(), torch.argmax(q, dim=-1)), f"{label}: action is not the first argmax of Q"
        diff = act.long() != torch.argmax(q64, dim=-1)
        bad = diff & ~_in_band(q64, bound)
        assert not bad.any(), f"{label}: {int(bad.sum())} greedy actions differ from argmax Q64 outside the band"
        flips = int(diff.sum())
        assert flips <= FLIP_SHARE * diff.numel(), f"{label}: {flips} excused argmax flips"
    return err, err32, flips


def _pair_contact(pos):
    """bool[B,N,N]: centre distance <= 2 r (the force of vmas' constraint is non-zero), diagonal excluded; float32
    norms like the oracle, with a one-ulp margin so that no borderline pair counts as contact-free."""
    from oracle import swarm_oracle as so
    B, N, _ = pos.shape
    d = torch.linalg.vector_norm(pos.unsqueeze(2) - pos.unsqueeze(1), dim=-1)
    c = d <= 2 * so.SPHERE_RADIUS * (1 + 1e-6)
    c[:, torch.arange(N), torch.arange(N)] = False
    return c


def _assert_close(name, got, ref, touched):
    """bit-exact where no contact force acted; STATE_RTOL (relative, with a 1e-1 floor of the denominator) elsewhere."""
    free = ~touched
    g, r = got[free], ref[free]
    assert torch.equal(g, r), f"{name}: {int((g != r).reshape(len(g), -1).any(-1).sum())} contact-free agents differ"
    g, r = got[touched].double(), ref[touched].double()
    if g.numel():
        err = ((g - r).abs() / r.abs().clamp_min(1e-1)).max().item()
        assert err <= STATE_RTOL, f"{name}: relative error {err:.3e} under contact"


def _check_world_step(label, scenario, s_in, actions, s_out, flags, rewards, keep=None):
    """The oracle's world step from (s_in, actions) against the kernel's post-step state / flags / rewards (envs in
    ``keep`` only).  Returns (touched agents, agent-agent contact of agent N-1)."""
    from oracle import batched_oracle as bo
    if keep is not None:
        s_in, actions, s_out, flags, rewards = s_in[keep], actions[keep], s_out[keep], flags[keep], rewards[keep]
    pos, vel = s_in[..., :2].contiguous(), s_in[..., 2:].contiguous()
    ref = bo.step(scenario, pos, vel, actions.long())
    pc = _pair_contact(pos)
    touched = pc.any(dim=2) | ((ref["flags"] & 1) != 0)
    assert torch.equal(flags, ref["flags"]), f"{label}: flags differ"
    _assert_close(f"{label} pos", s_out[..., :2], ref["pos"], touched)
    _assert_close(f"{label} vel", s_out[..., 2:], ref["vel"], touched)
    rt = touched if scenario == "obstacle_avoidance" else touched.any(dim=1, keepdim=True).expand_as(touched)
    _assert_close(f"{label} rewards", rewards, ref["rewards"], rt)
    return touched, pc[:, -1].any(dim=1)


def _rollout_vs_oracle(scenario, N, B, T, graph, params, label, bound=Q_BOUND):
    """Part 1 on one shape: generic traced rollout, every tick judged on its own input state."""
    sb = _sb()
    ops = sb.ops
    cfg = ops.make_config(_scen(scenario), B, N, _gmode(graph), 5, 0.35)
    s0 = _random_states(scenario, B, N, seed=1000 * N + B)
    out = ops.rollout(cfg, sb.pack_weights(params, _dev()), s0.to(_dev()), T,
                      trace=dict(state=True, actions=True, q=True, rewards=True, flags=True))
    tr = {k: out["trace_" + k].cpu() for k in ("state", "actions", "q", "rewards", "flags")}
    worst = worst32 = 0.0
    flips = 0
    touched_any = last_any = False
    for t in range(T):
        s_in = s0 if t == 0 else tr["state"][t - 1]
        q64, q32 = _oracle_q(params, s_in, graph)
        e, e32, f = _check_q(f"{label} t{t}", tr["q"][t], q64, q32, tr["actions"][t], bound)
        worst, worst32, flips = max(worst, e), max(worst32, e32), flips + f
        touched, last = _check_world_step(f"{label} t{t}", scenario, s_in, tr["actions"][t], tr["state"][t],
                                          tr["flags"][t], tr["rewards"][t])
        touched_any |= bool(touched.any())
        last_any |= bool(last.any())
    assert touched_any and last_any, f"{label}: the inputs should exercise contacts, including agent N-1's"
    assert torch.equal(out["state"].cpu(), tr["state"][T - 1])
    ret = torch.zeros(B, N)
    for t in range(T):
        ret = ret + tr["rewards"][t]
    assert torch.equal(out["returns"].cpu(), ret), f"{label}: returns != tick-ordered sum of the traced rewards"
    assert torch.equal(out["hits"].cpu().long(), ((tr["flags"] & 2) != 0).sum(dim=(0, 2))), f"{label}: hits"
    print(f"{label}: Q err vs float64 {worst:.2e} (float32 oracle {worst32:.2e}), excused flips {flips}")
    return worst


# N = 12 (epb = 10; the rollout takes the NT = 12 instantiation)
N12_CASES = [
    # 444 CTAs: 256 of 2 envs, 188 of 1 (3-CTA build)
    ("obstacle_avoidance", "complete", 700, 0),
    # 444 CTAs of 9-10 envs (3-CTA build): the benchmark shape
    ("obstacle_avoidance", "complete", 4096, 1),
    # DENSE: 592 CTAs of 8-9 envs
    ("obstacle_avoidance", "complete", 5000, 2),
    # DENSE, uniform packing: 600 CTAs of 10 envs and a last CTA of 7
    ("obstacle_avoidance", "complete", 6007, 3),
    # DENSE, balanced (592 CTAs of 8-9 envs), GoTo's collective reward
    ("go_to", "complete", 5000, 4),
    # 444 CTAs of 9-10 envs, kNN k = 5: ATT_COUNTS with the memo table
    ("obstacle_avoidance", "knn", 4096, 5),
    # 444 CTAs of 9-10 envs, radius 0.35: ATT_LIST
    ("go_to", "radius", 4096, 6),
]


@pytest.mark.parametrize("scenario,graph,B,model", N12_CASES)
def test_rollout_per_tick_oracle_n12(scenario, graph, B, model):
    _rollout_vs_oracle(scenario, 12, B, 8, graph, load_params(_exp(scenario), model), f"N12 {graph} B{B} {scenario}")


# run-time N, complete graph (epb = floor(128 / N)); B about 0.9 x 444 x epb, so that every CTA holds several envs
SWEEP = [
    (2, 25000, 3),    # 444 CTAs of 56-57 envs (epb 64)
    (3, 16000, 3),    # 444 CTAs of 36-37 (epb 42, 2 idle threads)
    (5, 10000, 3),    # 444 CTAs of 22-23 (epb 25, 3 idle threads)
    (7, 7000, 3),     # 444 CTAs of 15-16 (epb 18, 2 idle threads)
    (9, 5000, 2),     # 444 CTAs of 11-12 (epb 14, 2 idle threads)
    (16, 3200, 2),    # 444 CTAs of 7-8 (epb 8)
    (33, 1200, 2),    # 444 CTAs of 2-3 (epb 3, 29 idle threads)
    (43, 1000, 2),    # DENSE: 592 CTAs of 1-2 (epb 2, 42 idle threads)
    (64, 800, 2),     # 444 CTAs of 1-2 (epb 2)
    (100, 40, 2),     # 40 CTAs of one env, 28 idle threads
    (128, 40, 2),     # 40 CTAs of one env, every thread busy
]


@pytest.mark.parametrize("N,B,T", SWEEP)
def test_rollout_per_tick_oracle_sweep(N, B, T):
    scenario = "obstacle_avoidance" if N % 2 else "go_to"
    _rollout_vs_oracle(scenario, N, B, T, "complete", load_params(_exp(scenario), N % 10), f"N{N} B{B} {scenario}")


def _forward_vs_oracle(scenario, N, B, params, label, bound=Q_BOUND):
    sb = _sb()
    cfg = sb.ops.make_config(_scen(scenario), B, N, sb._lib.GRAPH_COMPLETE)
    st = _random_states(scenario, B, N, seed=7 * N + B)
    q, act = sb.ops.gatq_forward(cfg, sb.pack_weights(params, _dev()), st.to(_dev()))
    q64, q32 = _oracle_q(params, st, "complete")
    e, e32, f = _check_q(label, q.cpu(), q64, q32, act.cpu(), bound)
    print(f"{label}: Q err vs float64 {e:.2e} (float32 oracle {e32:.2e}), excused flips {f}")


@pytest.mark.parametrize("N,B", [(12, 4096),     # MODE_FORWARD, run-time N: 444 CTAs of 9-10 envs
                                 (7, 7000),      # 444 CTAs of 15-16
                                 (33, 1200)])    # 444 CTAs of 2-3
def test_forward_oracle(N, B):
    _forward_vs_oracle("obstacle_avoidance", N, B, load_params("ObstacleAvoidance", 8), f"forward N{N} B{B}")


def _plain_step_vs_oracle(scenario, N, B, params, label, bound=Q_BOUND):
    """Part 2: states of a generic rollout at ticks 0, 10, 30 and 60; one untraced tick from each (at N = 12 the PLAIN
    instantiation) with non-zero returns / hits going in, against the float32 oracle's greedy step."""
    from oracle import swarm_oracle as so, batched_oracle as bo
    sb = _sb()
    ops = sb.ops
    w = sb.pack_weights(params, _dev())
    cfg = ops.make_config(_scen(scenario), B, N, sb._lib.GRAPH_COMPLETE)
    g = torch.Generator().manual_seed(B + N)
    centers = torch.stack([so.draw_center(scenario, True, g) for _ in range(B)])
    if scenario == so.OBSTACLE_AVOIDANCE:           # a third of the swarms start on the obstacle: contacts
        centers[::3] = torch.tensor(list(so.OBSTACLE_POS)) + 0.1 * torch.randn(len(centers[::3]), 2, generator=g)
    s0 = ops.reset_grid(cfg, centers.to(_dev()))
    run = ops.rollout(cfg, w, s0.clone(), 60, trace=dict(state=True))
    states = [s0.cpu()] + [run["trace_state"][t - 1].cpu() for t in (10, 30, 60)]
    skipped = total = 0
    contact = False
    for k, S in enumerate(states):
        ret0 = torch.randn(B, N, generator=g)
        hits0 = torch.randint(0, 1000, (B,), generator=g, dtype=torch.int32)
        out = ops.rollout(cfg, w, S.to(_dev()), 1, returns=ret0.to(_dev()), hits=hits0.to(_dev()))
        got_s, got_r, got_h = out["state"].cpu(), out["returns"].cpu(), out["hits"].cpu().long()
        q64, q32 = _oracle_q(params, S, "complete")
        assert torch.isfinite(q64).all()
        act = torch.argmax(q32, dim=-1)
        keep = ~_in_band(q64, bound).any(dim=1)
        assert torch.equal(act[keep], torch.argmax(q64, dim=-1)[keep]), f"{label}: float32 oracle argmax off Q64"
        skipped += int((~keep).sum())
        total += B
        S, act, got_s, got_r, got_h, ret0, hits0 = (v[keep] for v in (S, act, got_s, got_r, got_h, ret0, hits0))
        pos = S[..., :2].contiguous()
        ref = bo.step(scenario, pos, S[..., 2:].contiguous(), act)
        touched = _pair_contact(pos).any(dim=2) | ((ref["flags"] & 1) != 0)
        contact |= bool(touched.any())
        _assert_close(f"{label} s{k} pos", got_s[..., :2], ref["pos"], touched)
        _assert_close(f"{label} s{k} vel", got_s[..., 2:], ref["vel"], touched)
        rt = touched if scenario == "obstacle_avoidance" else touched.any(dim=1, keepdim=True).expand_as(touched)
        _assert_close(f"{label} s{k} returns", got_r, ret0 + ref["rewards"], rt)
        assert torch.equal(got_h, hits0.long() + ((ref["flags"] & 2) != 0).sum(dim=1)), f"{label} s{k}: hits"
    assert skipped <= SKIP_SHARE * total, f"{label}: {skipped} / {total} envs skipped (in-band agents)"
    if B >= 48:
        assert contact, f"{label}: the states should exercise contacts"
    print(f"{label}: {skipped} / {total} envs skipped")


@pytest.mark.parametrize("scenario", ["obstacle_avoidance", "go_to"])
@pytest.mark.parametrize("B", [1,         # one CTA, one env: 116 inactive threads compute on env 0
                               48,        # 48 CTAs of one env
                               4096,      # 444 CTAs of 9-10 envs (3-CTA build)
                               5000,      # DENSE, 592 CTAs of 8-9
                               6007])     # DENSE, 600 CTAs of 10 and a last CTA of 7
def test_plain_step_oracle(scenario, B):
    _plain_step_vs_oracle(scenario, 12, B, load_params(_exp(scenario), 2), f"plain B{B} {scenario}")


# ---- part 3: stretched logits ------------------------------------------------------------------------------------
def _stretched_oa():
    """ObstacleAvoidance model 6 with conv1.att_src / att_dst x STRETCH: its attention leans on the agent id, so the
    last agent's logit leads many rows by more than 88.7 -- exp of that lead overflows float32, which only the
    softmax shift prevents."""
    return _stretched(load_params("ObstacleAvoidance", 6))


def _assert_stretched(params, state):
    """The precondition of part 3 on the inputs actually used: in-env logit spreads of at least 100 (median), and rows
    whose largest logit (agent N-1's) leads the rest by more than log(FLT_MAX)."""
    from oracle import batched_oracle as bo
    N = state.shape[1]
    x = bo.node_features(state[..., :2], state[..., 2:]).double()
    h = x @ params["conv1.lin.weight"].double().t()
    a_s = h @ params["conv1.att_src"].double().reshape(-1)
    a_d = h @ params["conv1.att_dst"].double().reshape(-1)
    z = a_s.unsqueeze(1) + a_d.unsqueeze(2)                             # [B, i, j]: logit of the edge j -> i
    z = torch.where(z > 0, z, 0.2 * z)
    eye = torch.eye(N, dtype=torch.bool)
    spread = z.masked_fill(eye, float("-inf")).amax(-1) - z.masked_fill(eye, float("inf")).amin(-1)
    lead = z[..., N - 1] - z.masked_fill(eye, float("-inf"))[..., :N - 1].amax(-1)
    assert spread.median().item() >= 100, f"logit spread {spread.median().item():.0f}"
    assert int((lead > 88.8).sum()) > 0, "no row where the last agent's logit leads by more than log(FLT_MAX)"


@pytest.mark.parametrize("N,B,T", [(12, 4096, 8),    # NT = 12: 444 CTAs of 9-10 envs
                                   (7, 7000, 3)])    # run-time N: 444 CTAs of 15-16
def test_stretched_rollout_per_tick_oracle(N, B, T):
    params = _stretched_oa()
    _assert_stretched(params, _random_states("obstacle_avoidance", B, N, seed=1000 * N + B)[:512])
    _rollout_vs_oracle("obstacle_avoidance", N, B, T, "complete", params, f"stretched N{N} B{B}", Q_BOUND_STRETCHED)


@pytest.mark.parametrize("N,B", [(12, 4096),         # PLAIN: 444 CTAs of 9-10 envs
                                 (7, 7000)])         # run-time N, untraced: 444 CTAs of 15-16
def test_stretched_plain_step_oracle(N, B):
    _plain_step_vs_oracle("obstacle_avoidance", N, B, _stretched_oa(), f"stretched plain N{N} B{B}", Q_BOUND_STRETCHED)


def test_stretched_forward_oracle():
    """MODE_FORWARD at N = 33 (444 CTAs of 2-3 envs)."""
    params = _stretched_oa()
    _assert_stretched(params, _random_states("obstacle_avoidance", 64, 33, seed=0))
    _forward_vs_oracle("obstacle_avoidance", 33, 1200, params, "stretched forward N33 B1200", Q_BOUND_STRETCHED)
