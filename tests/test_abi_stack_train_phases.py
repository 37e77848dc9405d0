"""Argument validation of the stacked train tick's two phases (swarm_train_tick_stack_grad / swarm_train_tick_stack_apply),
without a device.  The grad phase must refuse every call swarm_train_tick_stack refuses, with the same code and message,
and then check its peer exchange; the apply phase refuses every cfg, spec and hyper-parameter set the tick refuses.  As
in test_abi_rejections.py the calls run in a child process that sees no CUDA device, with a fake address wherever a call
needs a non-NULL pointer: a call that wrongly got past its checks fails with SWARM_ERR_CUDA instead of launching."""
import ctypes as C
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

P = 8              # a fake device address
BIG = 1 << 40      # a workspace size no check refuses
NAN = float("nan")

# rejections shared by swarm_train_tick_stack and swarm_train_tick_stack_grad: (id, call arguments, code, message fragment)
SHARED = [
    ("cfg_null", dict(c=None), -1, "cfg is NULL"),
    ("hyper_null", dict(h=None), -1, "hyper is NULL"),
    ("spec_null", dict(s=None), -1, "spec is NULL"),
    ("spec_layers", dict(s=dict(n_layers=5)), -1, "n_layers"),
    ("spec_hidden", dict(s=dict(hidden=33)), -2, "hidden"),
    ("spec_in_features", dict(s=dict(in_features=3)), -1, "in_features"),
    ("spec_activation", dict(s=dict(act=[0, 7, 1])), -1, "unknown activation"),
    ("agents_129", dict(c=dict(n=129)), -2, "n_agents > 128"),
    ("agents_1", dict(c=dict(n=1)), -2, "n_agents >= 2"),
    ("knn_above_16", dict(c=dict(n=20, graph="knn", k=5)), -2, "n_agents <= 16"),
    ("num_envs", dict(c=dict(B=0)), -1, "num_envs must be positive"),
    ("hyper_first", dict(c=dict(B=0), h=dict(graphs_per_update=0)), -1, "graphs_per_update"),
    ("update_target_every", dict(h=dict(update_target_every=0)), -1, "update_target_every"),
    ("adam_lr", dict(h=dict(lr=-1.0)), -1, "Adam"),
    ("adam_beta1", dict(h=dict(beta1=1.0)), -1, "Adam"),
    ("adam_beta2", dict(h=dict(beta2=-0.1)), -1, "Adam"),
    ("adam_eps", dict(h=dict(eps=NAN)), -1, "Adam"),
    ("hyper_flocking", dict(h="flocking"), -1, "hyper->flocking"),
    ("null_ctl", dict(null="ctl"), -1, "NULL argument"),
    ("null_weights", dict(null="weights"), -1, "NULL argument"),
    ("null_target", dict(null="target"), -1, "NULL argument"),
    ("null_state", dict(null="state"), -1, "NULL argument"),
    ("null_grad", dict(null="grad"), -1, "NULL argument"),
    ("null_workspace", dict(null="workspace"), -1, "NULL argument"),
    ("null_first", dict(null="ctl", r=dict(state=None)), -1, "NULL argument"),
    ("ring_null", dict(r=dict(state=None)), -1, "replay ring has NULL arrays"),
    ("ring_capacity", dict(r=dict(cap=0)), -1, "no capacity"),
    ("ring_below_num_envs", dict(r=dict(cap=63)), -1, "num_envs exceeds the replay capacity"),
    ("workspace", dict(wsb=16), -1, "workspace too small"),
    ("reward_kind", dict(reward=dict(kind=9)), -1, "unknown reward kind"),
    ("reward_disagree", dict(reward=dict(kind="cohesion", B=65)), -1, "disagree"),
    ("reward_world", dict(c=dict(scenario="oa"), reward=dict(kind="cohesion")), -1, "GoTo world"),
    ("reward_sigma", dict(reward=dict(kind="cohesion", sigma=NAN)), -1, "sigma"),
    ("reward_shaping", dict(reward=dict(kind="flocking"), shaping=None), -1, "shaping"),
    ("workspace_before_reward", dict(wsb=16, reward=dict(kind=9)), -1, "workspace too small"),
]

# swarm_train_tick_stack_grad only: the peer exchange, checked after everything the tick checks
PEERS = [
    ("peers_world_0", dict(peers=(0, 0, True)), -1, "peer exchange: bad world_size / rank"),
    ("peers_world_17", dict(peers=(17, 0, True)), -1, "peer exchange: bad world_size / rank"),
    ("peers_rank_high", dict(peers=(2, 2, True)), -1, "peer exchange: bad world_size / rank"),
    ("peers_rank_negative", dict(peers=(2, -1, True)), -1, "peer exchange: bad world_size / rank"),
    ("peers_null_buffer", dict(peers=(2, 1, False)), -1, "peer exchange: NULL peer buffer"),
    ("peers_after_tick_checks", dict(peers=(0, 0, True), wsb=16), -1, "workspace too small"),
]

# swarm_train_tick_stack_apply
APPLY = [
    ("cfg_null", dict(c=None), -1, "cfg is NULL"),
    ("hyper_null", dict(h=None), -1, "hyper is NULL"),
    ("spec_null", dict(s=None), -1, "spec is NULL"),
    ("spec_layers", dict(s=dict(n_layers=5)), -1, "n_layers"),
    ("spec_hidden", dict(s=dict(hidden=0)), -2, "hidden"),
    ("agents_129", dict(c=dict(n=129)), -2, "n_agents > 128"),
    ("agents_1", dict(c=dict(n=1)), -2, "n_agents >= 2"),
    ("knn_above_16", dict(c=dict(n=20, graph="knn", k=5)), -2, "n_agents <= 16"),
    ("num_envs", dict(c=dict(B=0)), -1, "num_envs must be positive"),
    ("graphs_per_update", dict(h=dict(graphs_per_update=0)), -1, "graphs_per_update"),
    ("adam_beta1", dict(h=dict(beta1=1.0)), -1, "Adam"),
    ("adam_eps", dict(h=dict(eps=-1.0)), -1, "Adam"),
    ("hyper_flocking", dict(h="flocking"), -1, "hyper->flocking"),
    ("null_ctl", dict(null="ctl"), -1, "NULL argument"),
    ("null_weights", dict(null="weights"), -1, "NULL argument"),
    ("null_target", dict(null="target"), -1, "NULL argument"),
    ("null_exp_avg", dict(null="exp_avg"), -1, "NULL argument"),
    ("null_exp_avg_sq", dict(null="exp_avg_sq"), -1, "NULL argument"),
    ("null_grad", dict(null="grad"), -1, "NULL argument"),
    ("ring_below_num_envs", dict(cap=63), -1, "num_envs exceeds the replay capacity"),
    ("null_first", dict(null="grad", cap=0), -1, "NULL argument"),
]


def _args(kw):
    """The C arguments of one case: cfg, spec, hyper, reward (+ the objects they point to, kept alive)."""
    import swarm_b200 as sb
    L, ops = sb._lib, sb.ops
    keep = []
    c = kw.get("c", {})
    cfg = None
    if c is not None:
        graph = {"complete": L.GRAPH_COMPLETE, "knn": L.GRAPH_KNN}[c.get("graph", "complete")]
        scen = L.SCENARIO_OBSTACLE_AVOIDANCE if c.get("scenario") == "oa" else L.SCENARIO_GOTO
        cfg = ops.make_config(scen, c.get("B", 64), c.get("n", 12), graph, c.get("k", 10))
        keep.append(cfg)
    s = kw.get("s", {})
    spec = None
    if s is not None:
        spec = ops.stack_spec(3, 8, 7)
        spec.n_layers = s.get("n_layers", 3)
        spec.hidden = s.get("hidden", 8)
        spec.in_features = s.get("in_features", 7)
        for i, a in enumerate(s.get("act", [])):
            spec.activation[i] = a
        keep.append(spec)
    h = kw.get("h", {})
    hyper = None
    if h is not None:
        hyper = L.SwarmTrainHyper()
        hyper.lr, hyper.beta1, hyper.beta2, hyper.eps, hyper.max_norm = 1e-3, 0.9, 0.999, 1e-8, 1.0
        hyper.graphs_per_update, hyper.update_target_every, hyper.gamma, hyper.loss_scale = 32, 200, 0.99, 1.0
        if h == "flocking":
            fs = ops.reward_spec(L.REWARD_FLOCKING, 64, 12)
            keep.append(fs)
            hyper.flocking, hyper.flocking_shaping = C.addressof(fs), P
        else:
            for k, v in h.items():
                setattr(hyper, k, v)
        keep.append(hyper)
    rw = kw.get("reward")
    reward = None
    if rw is not None:
        kind = {"flocking": L.REWARD_FLOCKING, "cohesion": L.REWARD_COHESION}.get(rw["kind"], rw["kind"])
        reward = ops.reward_spec(L.REWARD_FLOCKING, rw.get("B", 64), 12)
        reward.kind = kind
        if "sigma" in rw:
            reward.sigma = rw["sigma"]
        keep.append(reward)
    ref = lambda o: C.byref(o) if o is not None else None
    return ref(cfg), ref(spec), ref(hyper), (C.addressof(reward) if reward is not None else None), keep


def _ring(kw):
    import swarm_b200 as sb
    r = kw.get("r", {})
    return sb._lib.SwarmReplay(r.get("state", P), P, P, P, r.get("cap", 1000))


def _ptr(kw, name):
    return None if kw.get("null") == name else P


def _tick(lib, kw):
    cfg, spec, hyper, reward, keep = _args(kw)
    ring = _ring(kw)
    p = lambda n: _ptr(kw, n)
    return lib.swarm_train_tick_stack(cfg, spec, hyper, reward, kw.get("shaping", P), p("ctl"), p("weights"), p("target"),
                                      p("exp_avg"), p("exp_avg_sq"), p("state"), None, None, C.byref(ring), None,
                                      p("grad"), p("workspace"), kw.get("wsb", BIG), None)


def _grad(lib, kw):
    import swarm_b200 as sb
    cfg, spec, hyper, reward, keep = _args(kw)
    ring = _ring(kw)
    p = lambda n: _ptr(kw, n)
    peers = None
    if "peers" in kw:
        world, rank, buffers = kw["peers"]
        px = sb._lib.SwarmPeerExchange()
        px.world_size, px.rank = world, rank
        for i in range(16):
            px.data[i] = P if buffers or i != world - 1 else None
        peers = C.byref(px)
    return lib.swarm_train_tick_stack_grad(cfg, spec, hyper, reward, kw.get("shaping", P), p("ctl"), p("weights"),
                                           p("target"), p("state"), None, None, C.byref(ring), None, p("grad"),
                                           p("workspace"), kw.get("wsb", BIG), peers, None)


def _apply(lib, kw):
    cfg, spec, hyper, _, keep = _args(kw)
    p = lambda n: _ptr(kw, n)
    return lib.swarm_train_tick_stack_apply(cfg, spec, hyper, p("ctl"), p("weights"), p("target"), p("exp_avg"),
                                            p("exp_avg_sq"), p("grad"), kw.get("cap", 1000), None)


def _child_main():
    import swarm_b200 as sb
    lib = sb._lib.lib()
    out = {}
    run = lambda fn, kw: [int(fn(lib, kw)), lib.swarm_last_error().decode()]
    for name, kw, _, _ in SHARED:
        out[f"tick/{name}"] = run(_tick, kw)
        out[f"grad/{name}"] = run(_grad, kw)
    for name, kw, _, _ in PEERS:
        out[f"grad/{name}"] = run(_grad, kw)
    for name, kw, _, _ in APPLY:
        out[f"apply/{name}"] = run(_apply, kw)
    # well-formed calls get past every check and fail only at the (missing) device
    out["grad/valid"] = run(_grad, {})
    out["grad/valid_peers"] = run(_grad, dict(peers=(2, 1, True)))
    out["apply/valid"] = run(_apply, {})
    print(json.dumps(out))


@pytest.fixture(scope="module")
def results():
    import swarm_b200
    swarm_b200._build.build()
    code = (f"import sys; sys.path[:0] = {[ROOT, os.path.dirname(__file__)]!r}; import test_abi_stack_train_phases as t; "
            "t._child_main()")
    child = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                           capture_output=True, text=True)
    assert child.returncode == 0, child.stderr
    return json.loads(child.stdout.strip().splitlines()[-1])


def _check(results, prefix, table):
    failures = []
    for name, _, code, text in table:
        rc, msg = results[f"{prefix}/{name}"]
        if rc != code or text not in msg:
            failures.append(f"{prefix}/{name}: got ({rc}, {msg!r}), want ({code}, ...{text!r}...)")
    assert not failures, "\n".join(failures)


def test_grad_phase_refuses_what_the_tick_refuses(results):
    _check(results, "tick", SHARED)
    _check(results, "grad", SHARED)
    for name, _, _, _ in SHARED:
        assert results[f"grad/{name}"] == results[f"tick/{name}"], name     # same code, same message


def test_grad_phase_checks_its_peer_exchange(results):
    _check(results, "grad", PEERS)


def test_apply_phase_refuses_bad_cfg_spec_and_hyper_parameters(results):
    _check(results, "apply", APPLY)


def test_well_formed_phase_calls_pass_the_checks(results):
    import swarm_b200 as sb
    for name in ("grad/valid", "grad/valid_peers", "apply/valid"):
        assert results[name][0] == -3, (name, results[name])                 # SWARM_ERR_CUDA: no device
    # the stacked exchange slot holds the largest stack's gradient + loss (L = 4, width 32, 7 inputs), in 64-byte rows
    spec = sb.ops.stack_spec(4, 32, 7)
    assert int(sb._lib.lib().swarm_stack_weight_count(C.byref(spec))) + 1 == 5034 <= sb._lib.XCHG_STACK_STRIDE
    assert sb._lib.XCHG_STACK_STRIDE % 8 == 0
