"""The summation order `torch_row_sum_cascade` (csrc/swarm_device.cuh) emulates: torch's CPU sum / mean over a contiguous
float32 row of up to 4 095 elements, including the cascade of ATen's multi_row_sum (SumKernel.cpp: level_power =
max(4, CeilLog2(groups) / 4), so after every 16 groups of four 8-float vectors the level-0 accumulators are added into
level 1 and cleared, and the levels are folded back before row_sum adds its leftover chunks, partials and tail).  The
large-swarm Flocking reward's `.pow(2).mean(-1)` over the N - 1 partner distances (flocking_scenario.py:109-121,148-160)
goes through it, so the kernel must add in this order to stay bit-exact up to 4 096 agents.  This file pins the order
against torch for every row length 1 .. 4 095, and checks the argument validation of the large-swarm reward entry points
(rejected before any launch, so no device is needed)."""
import ctypes as C

import numpy as np
import torch

F = np.float32


def row_sum_cascade(e: np.ndarray, cascade: bool = True) -> np.ndarray:
    """Step-for-step twin of the device function (same variable names), vectorised over the rows of e f32[R, m].
    cascade = False leaves out the level-1 accumulators: the order of torch_row_sum."""
    R, m = e.shape
    if m < 8:
        p0 = p1 = p2 = p3 = np.zeros(R, F)
        k = 0
        if m >= 4:
            p0, p1, p2, p3 = e[:, 0], e[:, 1], e[:, 2], e[:, 3]
            k = 4
        for k in range(k, m):
            p0 = p0 + e[:, k]
        return ((p0 + p1) + p2) + p3
    chunks, groups = m >> 3, (m >> 3) >> 2
    a0, a1, a2, a3, b0, b1, b2, b3 = (np.zeros((R, 8), F) for _ in range(8))
    c = 0
    for gI in range(groups):
        a0 = a0 + e[:, (c + 0) * 8:(c + 1) * 8]
        a1 = a1 + e[:, (c + 1) * 8:(c + 2) * 8]
        a2 = a2 + e[:, (c + 2) * 8:(c + 3) * 8]
        a3 = a3 + e[:, (c + 3) * 8:(c + 4) * 8]
        if cascade and (gI & 15) == 15:                     # a full block of 16 groups: level 0 -> level 1
            b0, b1, b2, b3 = b0 + a0, b1 + a1, b2 + a2, b3 + a3
            a0, a1, a2, a3 = (np.zeros((R, 8), F) for _ in range(4))
        c += 4
    if cascade and groups >= 16:                            # level 1 -> level 0
        a0, a1, a2, a3 = a0 + b0, a1 + b1, a2 + b2, a3 + b3
    while c < chunks:
        a0 = a0 + e[:, c * 8:(c + 1) * 8]
        c += 1
    if groups > 0:
        a0 = ((a0 + a1) + a2) + a3
    fin = np.zeros(R, F)
    for k in range(chunks * 8, m):
        fin = fin + e[:, k]
    for l in range(8):
        fin = fin + a0[:, l]
    return fin


def test_row_sum_cascade_equals_torch_cpu_sum_and_mean_for_every_row_length():
    torch.set_num_threads(1)
    rng = np.random.default_rng(0)
    R = 3
    cascade_free_differs = 0
    for m in range(1, 4096):
        scale = (10.0 ** rng.integers(-3, 3, size=(R, 1))).astype(F)
        e = (rng.random((R, m), dtype=F) * scale).astype(F)
        got = row_sum_cascade(e)
        rows = torch.from_numpy(e)
        want = np.array([rows[r:r + 1].sum(-1).item() for r in range(R)], dtype=F)
        assert np.array_equal(got, want), f"m = {m}"
        # the same order when torch reduces several rows at once (the vectorised Flocking judge of the GPU tests)
        assert np.array_equal(rows.sum(-1).numpy(), want), f"m = {m}: multi-row sum"
        assert np.array_equal(rows.mean(-1).numpy(), (want / F(m)).astype(F)), f"m = {m}: mean = sum / count"
        cascade_free_differs += int((row_sum_cascade(e, cascade=False) != want).sum())
    # without the cascade about a third of the rows from 576 elements on come out different
    assert cascade_free_differs > 1000, "a cascade-free sum would be indistinguishable: the test would prove nothing"


def test_cascade_order_is_torch_row_sum_below_576_elements():
    rng = np.random.default_rng(1)
    for m in range(1, 576):
        e = rng.random((4, m), dtype=F)
        assert np.array_equal(row_sum_cascade(e), row_sum_cascade(e, cascade=False)), f"m = {m}"


# ---- argument errors of the large-swarm entry points (no device needed: rejected before any launch) -----------------
def _lib():
    import swarm_b200 as sb
    return sb._lib, sb._lib.lib(), sb.ops


def test_scenario_reward_large_argument_errors():
    L, lib, ops = _lib()
    FLOCK, COH = L.REWARD_FLOCKING, L.REWARD_COHESION

    def spec(kind=FLOCK, B=2, N=1024, **kw):
        sp = L.SwarmRewardSpec()
        lib.swarm_default_reward_spec(C.byref(sp), kind, B, N)
        for k, v in kw.items():
            setattr(sp, k, v)
        return sp

    ws = lambda sp: int(lib.swarm_scenario_reward_large_workspace_bytes(C.byref(sp)))       # noqa: E731

    def call(sp, state=8, shaping=8, reward=8, terms=None, workspace=8, wb=None):
        return lib.swarm_scenario_reward_large(C.byref(sp), state, shaping, reward, terms, workspace,
                                               ws(sp) if wb is None else wb, None)

    def err(rc, code, text):
        assert rc == code and text in lib.swarm_last_error(), (rc, lib.swarm_last_error())

    assert ws(spec()) == 2 * 1024 * 4 and ws(spec(COH)) == 0 and ws(spec(B=256, N=4096)) == 256 * 4096 * 4
    err(call(spec(N=1)), -1, b"at least two agents")
    err(call(spec(N=4097)), -2, b"n_agents <= 4096")
    assert ws(spec(N=4097)) == 0 and ws(spec(N=1)) == 0
    err(call(spec(), state=None), -1, b"state is NULL")
    err(call(spec(), shaping=None), -1, b"shaping")
    err(call(spec(), reward=None), -1, b"reward is NULL")
    err(call(spec(COH), reward=None), -1, b"reward is NULL")
    err(call(spec(COH, reset=1)), -1, b"reset must be 0")
    err(call(spec(COH, sigma=0.0)), -1, b"sigma must be > 0")
    err(call(spec(COH, sigma=-1.0)), -1, b"sigma must be > 0")
    err(call(spec(), wb=2 * 1024 * 4 - 1), -1, b"workspace too small")
    err(call(spec(), workspace=None), -1, b"workspace is NULL")
    err(call(spec(env_index=2)), -1, b"env_index out of range")
    err(call(spec(kind=7)), -1, b"unknown reward kind")
    err(call(spec(B=524288, N=4096)), -2, b"2^31")
    err(call(spec(B=(1 << 31) // 4096 - 1, N=4096, env_index=-1), state=None), -1, b"state is NULL")   # just below: accepted
    assert call(spec(B=0), state=None, shaping=None, reward=None, workspace=None, wb=0) == 0      # num_envs = 0: no-op
    assert call(spec(COH, B=0), state=None, shaping=None, reward=None, workspace=None, wb=0) == 0
    # reset needs no reward; a Cohesion call no workspace -- both still rejected here for the NULL state only
    err(call(spec(reset=1), state=None, reward=None), -1, b"state is NULL")
    err(call(spec(COH), state=None, workspace=None, wb=0), -1, b"state is NULL")
    # the env-tile entry point keeps its limit
    assert lib.swarm_scenario_reward(C.byref(spec(N=129)), 8, 8, 8, None, None) == -2


def test_rollout_stack_large_argument_errors():
    L, lib, ops = _lib()
    spec = ops.stack_spec(3, 8, 7)
    cfg = ops.make_config(L.SCENARIO_GOTO, 2, 1024, L.GRAPH_RADIUS)
    rs = L.SwarmRewardSpec()
    lib.swarm_default_reward_spec(C.byref(rs), L.REWARD_FLOCKING, 2, 1024)
    coh = L.SwarmRewardSpec()
    lib.swarm_default_reward_spec(C.byref(coh), L.REWARD_COHESION, 2, 1024)
    ws = lambda c, r=None: int(lib.swarm_rollout_stack_large_workspace_bytes(C.byref(c), C.byref(r) if r else None))  # noqa

    def call(c, r=None, shaping=8, wb=None):
        return lib.swarm_rollout_stack_large(C.byref(c), C.byref(spec), 8, 8, 1, C.byref(r) if r else None, shaping, 8, 8, 8,
                                             ws(c, r) if wb is None else wb, None)

    base = int(lib.swarm_rollout_stack_workspace_bytes(C.byref(cfg)))
    assert ws(cfg) == base
    assert ws(cfg, rs) == base + 256 + 2 * 1024 * 4 and ws(cfg, coh) == base + 256
    assert call(cfg, rs, wb=ws(cfg, rs) - 1) == -1 and b"workspace too small" in lib.swarm_last_error()
    assert call(cfg, rs, wb=base) == -1 and b"workspace too small" in lib.swarm_last_error()
    assert call(cfg, rs, shaping=None) == -1 and b"shaping" in lib.swarm_last_error()
    bad_sigma = L.SwarmRewardSpec.from_buffer_copy(coh)
    bad_sigma.sigma = 0.0
    assert call(cfg, bad_sigma) == -1 and b"sigma" in lib.swarm_last_error()
    other = L.SwarmRewardSpec.from_buffer_copy(rs)
    other.n_agents = 512
    assert call(cfg, other) == -1 and b"disagree" in lib.swarm_last_error()
    oa = ops.make_config(L.SCENARIO_OBSTACLE_AVOIDANCE, 2, 1024, L.GRAPH_RADIUS)
    assert call(oa, rs) == -1 and b"GoTo world" in lib.swarm_last_error()
    small = ops.make_config(L.SCENARIO_GOTO, 2, 128, L.GRAPH_RADIUS)
    assert ws(small) == 0 and call(small, wb=1 << 30) == -2 and b"swarm_rollout_stack" in lib.swarm_last_error()
    big = ops.make_config(L.SCENARIO_GOTO, 2, 4097, L.GRAPH_RADIUS)
    assert ws(big) == 0 and call(big, wb=1 << 30) == -2
    assert lib.swarm_rollout_stack_large(C.byref(cfg), C.byref(spec), 8, 8, -1, None, None, None, None, 8, base, None) == -1
    assert b"ticks" in lib.swarm_last_error()
    # swarm_rollout_stack keeps its answer above 128 agents
    assert lib.swarm_rollout_stack(C.byref(cfg), C.byref(spec), 8, 8, 1, C.byref(rs), 8, None, None, 8, base, None) == -2
