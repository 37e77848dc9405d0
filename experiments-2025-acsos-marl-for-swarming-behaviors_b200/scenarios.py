"""The VMAS scenario seam: ``World`` / ``Agent`` / ``Landmark`` / ``Sphere`` / ``Color`` / ``BaseScenario`` with the
constructor signatures and attributes of vmas==1.4.0 that scenario files are written against
(``vmas.simulator.core``, ``vmas.simulator.scenario``, ``vmas.simulator.utils``), plus the two scenarios of the
hot path, GoTo-position and ObstacleAvoidance.

Mirrors src/scenarios/go_to_position_scenario.py:7-149 and src/scenarios/obstacle_avoidance_scenario.py:7-181
(``make_world / reset_world_at / observation / reward / done / info`` plus the metric methods the Simulator calls on
``env.scenario``).  The arithmetic is not here: ``World.step`` runs ``swarm_sim_step`` on the world's
structure-of-arrays state, entities are views into it, and the two built-in scenarios return what the kernel wrote
for the agent they are asked about.

A scenario written by a user against the vmas API (its own ``make_world`` building ``World(batch_dim, device)``,
``Landmark(...)``, ``Agent(...)``; rewards / observations computed with torch from ``agent.state.pos``) runs on the
same CUDA world step as long as it stays inside what the kernels implement: sphere agents of one radius, at most one
colliding (sphere) landmark at a batch-constant position, vmas' default holonomic dynamics with discrete actions.
Anything else raises ``NotImplementedError`` at world construction -- there is no CPU fallback.
"""
from __future__ import annotations

import enum
from typing import Dict, List, Optional, Sequence

import torch

from . import _lib, ops


class Color(enum.Enum):
    """vmas.simulator.utils.Color (rendering only)."""
    RED = (0.75, 0.25, 0.25)
    GREEN = (0.25, 0.75, 0.25)
    BLUE = (0.25, 0.25, 0.75)
    LIGHT_GREEN = (0.45, 0.95, 0.45)
    WHITE = (0.75, 0.75, 0.75)
    GRAY = (0.25, 0.25, 0.25)
    BLACK = (0.15, 0.15, 0.15)


class Shape:
    pass


class Sphere(Shape):
    """vmas.simulator.core.Sphere; the default entity shape (radius 0.05)."""

    def __init__(self, radius: float = 0.05):
        if not radius > 0:
            raise AssertionError(f"Radius must be > 0, got {radius}")
        self.radius = float(radius)


class Box(Shape):
    def __init__(self, length: float = 0.3, width: float = 0.1, hollow: bool = False):
        self.length, self.width, self.hollow = length, width, hollow


class Line(Shape):
    def __init__(self, length: float = 0.5):
        self.length = length


class _EntityState:
    def __init__(self, pos: Optional[torch.Tensor], vel: Optional[torch.Tensor]):
        self.pos = pos
        self.vel = vel


class Entity:
    """Common part of vmas Agent / Landmark: name, collide / movable flags, shape, colour, batched state."""

    def __init__(self, name: str, movable: bool = False, rotatable: bool = False, collide: bool = True,
                 density: float = 25.0, mass: float = 1.0, shape: Optional[Shape] = None, v_range: Optional[float] = None,
                 max_speed: Optional[float] = None, color=Color.GRAY, is_joint: bool = False, drag: Optional[float] = None,
                 linear_friction: Optional[float] = None, angular_friction: Optional[float] = None, gravity=None,
                 collision_filter=None, **_ignored):
        self.name = name
        self.movable = movable
        self.rotatable = rotatable
        self.collide = collide
        self.mass = mass
        self.shape = shape if shape is not None else Sphere()
        self.color = color
        self.v_range, self.max_speed = v_range, max_speed
        if is_joint or drag is not None or linear_friction is not None or angular_friction is not None or gravity is not None:
            raise NotImplementedError("per-entity drag / friction / gravity / joints are outside the swarm_b200 kernels")
        self._world: Optional["World"] = None
        self._index: Optional[int] = None
        self._pos: Optional[torch.Tensor] = None          # landmarks own their position tensor
        self._host_pos: Optional[tuple] = None            # batch-constant position mirrored on the host (kernel constants)

    # vmas names
    @property
    def batch_dim(self) -> int:
        return self._world.batch_dim

    @property
    def device(self):
        return self._world.device

    def _require_world(self) -> "World":
        if self._world is None:
            raise AssertionError(f"{self.name} has not been added to a World")
        return self._world

    def _mirror(self) -> None:
        """Host-seam worlds (see World): what was just written into the host copy of this entity also goes to HBM."""

    def set_vel(self, vel: torch.Tensor, batch_index: Optional[int] = None) -> None:
        st = self.state
        if st.vel is None:
            return
        v = torch.as_tensor(vel, dtype=torch.float32).to(st.vel.device)
        if batch_index is None:
            st.vel[...] = v
        else:
            st.vel[batch_index] = v
        self._mirror()

    def set_pos(self, pos: torch.Tensor, batch_index: Optional[int] = None) -> None:
        st = self.state
        self._require_world().version += 1
        p_host = torch.as_tensor(pos, dtype=torch.float32)
        p = p_host.to(st.pos.device)
        # a 1-D position is one value for every env it is written to: mirrored on the host (kernel constant); a device
        # tensor costs one tiny D2H copy here, at reset time
        vec = tuple(float(v) for v in p_host.detach().cpu()[:2]) if p_host.dim() == 1 else None
        if batch_index is None:
            st.pos[...] = p
            self._host_pos = vec
        else:
            st.pos[batch_index] = p
            if self._world.batch_dim == 1 and vec is not None:
                self._host_pos = vec
            elif self._host_pos is not None and vec != self._host_pos:
                self._host_pos = None
        self._mirror()


class Landmark(Entity):
    """vmas.simulator.core.Landmark: static by default; ``collide=True`` makes it the obstacle of the world step."""

    def __init__(self, name: str, shape: Optional[Shape] = None, movable: bool = False, rotatable: bool = False,
                 collide: bool = True, density: float = 25.0, mass: float = 1.0, v_range=None, max_speed=None,
                 color=Color.GRAY, **kwargs):
        super().__init__(name, movable, rotatable, collide, density, mass, shape, v_range, max_speed, color, **kwargs)

    @property
    def state(self) -> _EntityState:
        self._require_world()
        return _EntityState(self._pos, None)


class Agent(Entity):
    """vmas.simulator.core.Agent: a view of one agent column of the world's SoA state."""

    def __init__(self, name: str, shape: Optional[Shape] = None, movable: bool = True, rotatable: bool = True,
                 collide: bool = True, density: float = 25.0, mass: float = 1.0, f_range=None, max_f=None, t_range=None,
                 max_t=None, v_range=None, max_speed=None, color=Color.BLUE, alpha: float = 0.5, obs_range=None,
                 obs_noise=None, u_noise=None, u_range: float = 1.0, u_multiplier: float = 1.0, action_script=None,
                 sensors=None, c_noise: float = 0.0, silent: bool = True, adversary: bool = False,
                 render_action: bool = False, dynamics=None, action_size=None, discrete_action_nvec=None, **kwargs):
        super().__init__(name, movable, rotatable, collide, density, mass, shape, v_range, max_speed, color, **kwargs)
        unsupported = {"f_range": f_range, "max_f": max_f, "obs_noise": obs_noise, "u_noise": u_noise,
                       "action_script": action_script, "sensors": sensors, "dynamics": dynamics,
                       "v_range": v_range, "max_speed": max_speed}
        bad = [k for k, v in unsupported.items() if v]
        if bad or u_range != 1.0 or u_multiplier != 1.0 or not movable or mass != 1.0:
            raise NotImplementedError(
                f"Agent({name}): {bad or 'u_range / u_multiplier / mass / movable'} differ from the vmas defaults the "
                "swarm_b200 world step implements (holonomic, mass 1, u_range 1, discrete 3 x 3 actions)")
        self.u_range, self.u_multiplier = u_range, u_multiplier
        self.render_action = render_action
        self.goal: Optional[Landmark] = None

    @property
    def index(self) -> int:
        return self._index

    @property
    def state(self) -> _EntityState:
        w = self._require_world()
        s = w.host_state if w.host_state is not None else w.state
        return _EntityState(s[:, self._index, 0:2], s[:, self._index, 2:4])

    def _mirror(self) -> None:
        w = self._world
        if w is not None and w.host_state is not None:
            w.state[:, self._index].copy_(w.host_state[:, self._index])


class World:
    """vmas.simulator.core.World with the state as one f32[B,N,4] tensor in HBM, stepped by the CUDA kernel."""

    def __init__(self, batch_dim: int, device, dt: float = 0.1, substeps: int = 1, drag: float = 0.25,
                 linear_friction: float = 0.0, angular_friction: float = 0.0, x_semidim: Optional[float] = None,
                 y_semidim: Optional[float] = None, dim_c: int = 0, collision_force: float = 100.0,
                 joint_force: float = 130.0, torque_constraint_force: float = 1.0, contact_margin: float = 1e-3,
                 gravity=(0.0, 0.0)):
        device = torch.device(device)
        compute = device
        if device.type != "cuda":
            # host-seam mode: the script asked for host tensors (the reference hard-codes device='cpu'); the world still
            # lives in HBM and is stepped by the CUDA kernel, entity states are read through a host copy refreshed
            # after every kernel (_lib.offload_device)
            compute = _lib.offload_device()
            if compute is None:
                raise _lib.SwarmError(f"swarm_b200 worlds live on a CUDA device (got {device}); there is no CPU fallback "
                                      "(set SWARM_DEVICE=cuda to serve a script that hard-codes device='cpu' from a B200)")
        if substeps != 1 or linear_friction or angular_friction or x_semidim is not None or y_semidim is not None or \
                tuple(float(g) for g in gravity) != (0.0, 0.0):
            raise NotImplementedError("substeps != 1, friction, world bounds and gravity are outside the swarm_b200 "
                                      "world step (the reference scenarios use the vmas defaults)")
        self.batch_dim = batch_dim
        self.device = device                   # where the script's tensors live (vmas World.device)
        self.compute_device = compute          # where the state lives and the kernels run
        self.host_state: Optional[torch.Tensor] = None
        self._dt, self._drag, self._collision_force, self._contact_margin = dt, drag, collision_force, contact_margin
        self._agents: List[Agent] = []
        self._landmarks: List[Landmark] = []
        self.state: Optional[torch.Tensor] = None
        self.cfg: Optional[_lib.SwarmConfig] = None
        self.last: Dict[str, torch.Tensor] = {}
        self._obstacle: Optional[Landmark] = None
        self._goal: Optional[Landmark] = None
        self.version = 0                       # bumped whenever the state may have changed (step / reset / set_pos)

    # vmas attribute names
    @property
    def agents(self) -> List[Agent]:
        return self._agents

    @property
    def landmarks(self) -> List[Landmark]:
        return self._landmarks

    @property
    def entities(self):
        return self._landmarks + self._agents

    @property
    def dt(self) -> float:
        return self._dt

    def add_agent(self, agent: Agent) -> None:
        if self.state is not None:
            raise AssertionError("agents must be added inside make_world")
        agent._world, agent._index = self, len(self._agents)
        self._agents.append(agent)

    def add_landmark(self, landmark: Landmark) -> None:
        landmark._world, landmark._index = self, len(self._landmarks)
        landmark._pos = torch.zeros(self.batch_dim, 2, dtype=torch.float32, device=self.device)
        landmark._host_pos = (0.0, 0.0)
        self._landmarks.append(landmark)

    def _finalize(self, scenario_id: Optional[int] = None) -> None:
        """Called once make_world has returned: freeze the entity set, check it against what the kernels implement,
        allocate the SoA state and derive the kernel configuration."""
        n = len(self._agents)
        if n == 0:
            raise AssertionError("a world needs at least one agent")
        radii = set()
        for a in self._agents:
            if not isinstance(a.shape, Sphere) or not a.collide:
                raise NotImplementedError("the swarm_b200 world step implements colliding sphere agents")
            radii.add(a.shape.radius)
        if len(radii) != 1:
            raise NotImplementedError("all agents must share one radius")
        obstacles = [l for l in self._landmarks if l.collide]
        if len(obstacles) > 1 or any(l.movable for l in self._landmarks):
            raise NotImplementedError("the swarm_b200 world step implements at most one colliding, static landmark")
        if obstacles and not isinstance(obstacles[0].shape, Sphere):
            raise NotImplementedError("the colliding landmark must be a sphere")
        self._obstacle = obstacles[0] if obstacles else None
        free = [l for l in self._landmarks if not l.collide]
        self._goal = free[0] if free else None
        if scenario_id is None:
            scenario_id = _lib.SCENARIO_OBSTACLE_AVOIDANCE if self._obstacle is not None else _lib.SCENARIO_GOTO
        cfg = ops.make_config(scenario_id, self.batch_dim, n)
        cfg.dt, cfg.drag = self._dt, self._drag
        cfg.collision_force, cfg.contact_margin = self._collision_force, self._contact_margin
        cfg.agent_radius = radii.pop()
        if self._obstacle is not None:
            cfg.landmark_radius = self._obstacle.shape.radius
        self.cfg = cfg
        self.state = torch.zeros(self.batch_dim, n, 4, dtype=torch.float32, device=self.compute_device)
        if self.compute_device != self.device:
            self.host_state = torch.zeros(self.batch_dim, n, 4, dtype=torch.float32).pin_memory()
        self._refresh_outputs()

    def _sync_constants(self) -> None:
        """Landmark positions are kernel constants (one value for all envs): mirror them into the config."""
        if self._obstacle is not None:
            if self._obstacle._host_pos is None:
                raise NotImplementedError("the obstacle must sit at the same position in every env")
            self.cfg.obstacle_x, self.cfg.obstacle_y = self._obstacle._host_pos
        if self._goal is not None:
            if self._goal._host_pos is None:
                raise NotImplementedError("the goal must sit at the same position in every env")
            self.cfg.goal_x, self.cfg.goal_y = self._goal._host_pos

    def _refresh_outputs(self) -> None:
        """Observation / distance terms of the current state without stepping (used after reset)."""
        B, N = self.cfg.num_envs, self.cfg.n_agents
        dev = self.compute_device
        goal = torch.tensor([self.cfg.goal_x, self.cfg.goal_y], dtype=torch.float32, device=dev)
        self.last = {
            "obs": torch.cat([self.state, goal.view(1, 1, 2).expand(B, N, 2)], dim=2),
            "rewards": torch.zeros(B, N, dtype=torch.float32, device=dev),
            "flags": torch.zeros(B, N, dtype=torch.uint8, device=dev),
            "dist": torch.zeros(B, N, 2, dtype=torch.float32, device=dev),
        }

    def _download(self) -> None:
        """Host-seam mode: refresh the host copy of the state after a kernel wrote it."""
        if self.host_state is not None:
            self.host_state.copy_(self.state)

    def reset(self, env_index: Optional[int] = None) -> None:
        """vmas World.reset: every entity's state back to zero (the scenario's reset_world_at places them next)."""
        self.version += 1
        if env_index is None:
            self.state.zero_()
        else:
            self.state[env_index].zero_()
        self._download()

    def reset_to_grid(self, centers: torch.Tensor, env_index: Optional[int] = None) -> None:
        """generate_grid + set_pos for every agent; velocities zero (vmas world.reset)."""
        centers = centers.to(device=self.compute_device, dtype=torch.float32).reshape(-1, 2)
        self.version += 1
        self._sync_constants()
        if env_index is None:
            if centers.shape[0] == 1:
                centers = centers.expand(self.batch_dim, 2)
            ops.reset_grid(self.cfg, centers.contiguous(), out=self.state)
        else:
            one = ops.clone_config(self.cfg, num_envs=1)
            ops.reset_grid(one, centers[:1].contiguous(), out=self.state[env_index])
        self._download()
        self._refresh_outputs()

    def step(self, actions: torch.Tensor) -> None:
        """actions int32[B,N] -> in-place world step; results kept in ``self.last``."""
        self._sync_constants()
        self.version += 1
        self.last = ops.sim_step(self.cfg, self.state, actions, state_out=self.state, want_obs=True)
        self._download()

    def adopt_rollout(self, out: Dict[str, torch.Tensor]) -> None:
        """A fused rollout (``ops.rollout``) advanced ``self.state`` in place: make the world look as it does after the
        last ``Environment.step`` of that rollout -- version bumped (version-keyed reward caches drop their entry) and
        ``self.last`` rebuilt from the last tick's traces, so that ``observation()`` / ``reward()`` /
        ``average_distance_to_goal()`` / ``obstacles_hits()`` report the final tick instead of the post-reset zeros.
        ``out`` must carry the ``rewards``, ``flags`` and ``dist`` traces."""
        B, N = self.cfg.num_envs, self.cfg.n_agents
        self.version += 1
        goal = torch.tensor([self.cfg.goal_x, self.cfg.goal_y], dtype=torch.float32, device=self.compute_device)
        self._download()
        self.last = {
            "state": self.state,
            "obs": torch.cat([self.state, goal.view(1, 1, 2).expand(B, N, 2)], dim=2),
            "rewards": out["trace_rewards"][-1].clone(),
            "flags": out["trace_flags"][-1].clone(),
            "dist": out["trace_dist"][-1].clone(),
        }

    def get_distance(self, a: Entity, b: Entity) -> torch.Tensor:
        """vmas World.get_distance for two spheres: centre distance minus the two radii (oa:149-150,168,171)."""
        if not isinstance(a.shape, Sphere) or not isinstance(b.shape, Sphere):
            raise NotImplementedError("get_distance is implemented for spheres")
        dist = torch.linalg.vector_norm(a.state.pos - b.state.pos, dim=-1)
        return dist - a.shape.radius - b.shape.radius


class BaseScenario:
    """vmas.simulator.scenario.BaseScenario: subclasses implement make_world / reset_world_at / observation / reward
    (and optionally done / info); the environment calls the ``env_*`` wrappers."""

    scenario_id: Optional[int] = None        # built-in scenarios name the fused reward kernel they use

    def __init__(self):
        self._world: Optional[World] = None

    @property
    def world(self) -> World:
        return self._world

    def to(self, device) -> None:            # vmas API; worlds are created on their device
        return None

    def env_make_world(self, batch_dim: int, device, **kwargs) -> World:
        self._world = self.make_world(batch_dim, device, **kwargs)
        if not isinstance(self._world, World):
            raise AssertionError("make_world must return a swarm_b200 World (vmas.simulator.core.World of the shim)")
        if self._world.state is None:
            self._world._finalize(self.scenario_id)
        return self._world

    def env_reset_world_at(self, env_index: Optional[int]) -> None:
        self.world.reset(env_index)
        self.reset_world_at(env_index)
        self.world._sync_constants()
        self.world._refresh_outputs()

    # -- to be provided by the scenario ---------------------------------------------------------------
    def make_world(self, batch_dim: int, device, **kwargs) -> World:
        raise NotImplementedError

    def reset_world_at(self, env_index: Optional[int] = None) -> None:
        raise NotImplementedError

    def observation(self, agent: Agent) -> torch.Tensor:
        raise NotImplementedError

    def reward(self, agent: Agent) -> torch.Tensor:
        raise NotImplementedError

    def done(self) -> torch.Tensor:
        return torch.zeros(self.world.batch_dim, device=self.world.device, dtype=torch.bool)

    def info(self, agent: Agent) -> Dict[str, torch.Tensor]:
        return {}

    def extra_render(self, env_index: int = 0):
        return []


class _KernelScenario(BaseScenario):
    """Shared part of the two hot-path scenarios: rewards, observations and metrics are what the fused world-step
    kernel wrote (bit-identical to the reference's per-agent torch code, see tests/test_gpu_parity.py)."""

    def _build_world(self, batch_dim: int, device, with_obstacle: bool) -> World:
        world = World(batch_dim, device)
        goal = Landmark(name="goal", collide=False, color=Color.BLACK)
        world.add_landmark(goal)
        if with_obstacle:
            world.add_landmark(Landmark(name="obstacle", collide=True, color=Color.RED))
        for i in range(self.n_agents):
            agent = Agent(name=f"agent{i}", collide=True, color=Color.GREEN, render_action=True)
            agent.pos_rew = torch.zeros(batch_dim, device=world.device)
            agent.collision_rew = agent.pos_rew.clone()
            agent.goal = goal
            world.add_agent(agent)
        world._finalize(self.scenario_id)
        self.pos_rew = torch.zeros(batch_dim, device=world.device)
        self.final_rew = self.pos_rew.clone()
        return world

    def observation(self, agent: Agent) -> torch.Tensor:
        """cat[pos, vel, goal] f32[B,6] (go_to:124-132, oa:154-162)."""
        return self.world.last["obs"][:, agent.index]

    def reward(self, agent: Agent) -> torch.Tensor:
        return self.world.last["rewards"][:, agent.index]

    def info(self, agent: Agent) -> Dict[str, torch.Tensor]:
        return {"pos_rew": agent.pos_rew, "final_rew": self.final_rew}

    def average_distance_to_goal(self) -> torch.Tensor:
        # torch.mean(torch.stack([agent.distance_to_goal ...])) (go_to:134-135) -- reduced on the host like the
        # reference (device = cpu there) so the metric is bit-identical; this is a per-tick metric read, not hot path
        return torch.mean(self.world.last["dist"][:, :, 0].cpu().transpose(0, 1).contiguous())

    def set_start_centers(self, centers: Optional[torch.Tensor]) -> None:
        """Batched extension: explicit per-env start centres f32[B,2] used by the next resets instead of
        the reference's single shared draw (SURVEY.md 7, hard part 3)."""
        self._explicit_centers = centers


class GoToPositionScenario(_KernelScenario):
    scenario_id = _lib.SCENARIO_GOTO

    def make_world(self, batch_dim: int, device, **kwargs) -> World:
        self.pos_shaping_factor = kwargs.get("pos_shaping_factor", 1.0)
        self.agent_radius = kwargs.get("agent_radius", 0.1)      # unused by the physics (SURVEY 7.6)
        self.n_agents = kwargs.get("n_agents", 1)
        self.seed = kwargs.get("seed", 1)
        self.per_env_centers = kwargs.get("per_env_centers", False)
        self._explicit_centers = None
        self.desired_distance = 0.15
        torch.manual_seed(self.seed)                              # go_to:23 (make_env never forwards `seed`)
        if torch.cuda.is_available():
            torch.cuda.manual_seed_all(self.seed)
        return self._build_world(batch_dim, device, with_obstacle=False)

    def reset_world_at(self, env_index: Optional[int] = None) -> None:
        w = self.world
        w.landmarks[0].set_pos(torch.tensor([-0.8, 0.8]), batch_index=env_index)        # go_to:86
        if self._explicit_centers is not None:
            centers = self._explicit_centers if env_index is None else self._explicit_centers[env_index:env_index + 1]
        else:
            n = w.batch_dim if (self.per_env_centers and env_index is None) else 1
            position_range = -torch.tensor([-1.5, 1.5])            # go_to:84-88
            if n == 1:
                centers = position_range + torch.normal(mean=torch.tensor([-0.6, 0.6]), std=torch.tensor([0.4, 0.4]))
            else:
                centers = position_range + torch.normal(mean=torch.tensor([-0.6, 0.6]).expand(n, 2),
                                                        std=torch.tensor([0.4, 0.4]).expand(n, 2))
        w.reset_to_grid(centers, env_index)

    def average_distance_to_obstacles(self) -> torch.Tensor:
        return torch.tensor(0.0)

    def obstacles_hits(self) -> torch.Tensor:
        return torch.tensor(0.0)


class ObstacleAvoidanceScenario(_KernelScenario):
    scenario_id = _lib.SCENARIO_OBSTACLE_AVOIDANCE

    def make_world(self, batch_dim: int, device, **kwargs) -> World:
        self.random = kwargs.get("random", False)
        self.pos_shaping_factor = kwargs.get("pos_shaping_factor", 10.0)
        self.dist_shaping_factor = kwargs.get("dist_shaping_factor", 10.0)
        self.agent_radius = kwargs.get("agent_radius", 0.1)
        self.n_agents = kwargs.get("n_agents", 1)
        self.per_env_centers = kwargs.get("per_env_centers", False)
        self._explicit_centers = None
        self.n_obstacles = 1
        self.desired_distance = 0.15
        self.min_collision_distance_reward = 1
        self.min_collision_distance_count = 0.2
        return self._build_world(batch_dim, device, with_obstacle=True)

    def reset_world_at(self, env_index: Optional[int] = None) -> None:
        w = self.world
        w.landmarks[0].set_pos(torch.tensor([-0.8, 0.8]), batch_index=env_index)        # oa:97
        w.landmarks[1].set_pos(torch.tensor([-0.1, 0.1]), batch_index=env_index)        # oa:99
        if self._explicit_centers is not None:
            centers = self._explicit_centers if env_index is None else self._explicit_centers[env_index:env_index + 1]
        else:
            n = w.batch_dim if (self.per_env_centers and env_index is None) else 1
            if self.random and n == 1:                             # oa:100-102
                delta = torch.normal(mean=torch.tensor([0.0, 0.0]), std=torch.tensor([0.1, 0.1]))
            elif self.random:
                delta = torch.normal(mean=torch.tensor([0.0, 0.0]).expand(n, 2), std=torch.tensor([0.1, 0.1]).expand(n, 2))
            else:
                delta = torch.zeros(n, 2)
            centers = torch.tensor([0.6, -0.6]) + delta
        w.reset_to_grid(centers, env_index)

    def average_distance_to_obstacles(self) -> torch.Tensor:
        return torch.mean(self.world.last["dist"][:, :, 1].cpu().transpose(0, 1).contiguous())

    def obstacles_hits(self) -> torch.Tensor:
        hits = (self.world.last["flags"] & _lib.FLAG_HIT) != 0       # oa:170-173
        return torch.sum(hits)


class FlockingScenario(BaseScenario):
    """src/scenarios/flocking_scenario.py:7-205.  The world is GoTo's (goal landmark that does not collide, colliding
    sphere agents) and is stepped by ``swarm_sim_step``; the collective reward -- shaped goal progress, +50 on the goal,
    -1 per near-contact, shaped spacing progress, with the two ``previous_*`` memories per agent -- is one
    ``swarm_scenario_reward`` launch per tick over all envs.  The reference branches on tensors in Python
    (flocking:141,169) and so only runs with ``num_envs = 1``; here every env is its own copy of that computation.
    Swarms of 2 to 4 096 agents: above 128 agents the reward runs through ``swarm_scenario_reward_large``."""

    scenario_id = _lib.SCENARIO_GOTO

    def make_world(self, batch_dim: int, device, **kwargs) -> World:
        self.pos_shaping_factor = kwargs.get("pos_shaping_factor", 10.0)
        self.dist_shaping_factor = kwargs.get("dist_shaping_factor", 10.0)
        self.agent_radius = kwargs.get("agent_radius", 0.1)       # unused by the physics, as in the reference
        self.n_agents = kwargs.get("n_agents", 1)
        self.per_env_centers = kwargs.get("per_env_centers", False)
        self._explicit_centers = None
        self.min_distance_between_entities = self.agent_radius * 2 + 0.05
        self.world_semidim = 1
        self.collective_reward = 0
        self.agent_collision_reward = -1
        self.desired_distance = 0.15
        self.min_collision_distance = 0.005

        world = World(batch_dim, device)
        goal = Landmark(name="goal", collide=False, color=Color.BLACK)
        world.add_landmark(goal)
        for i in range(self.n_agents):
            agent = Agent(name=f"agent{i}", collide=True, color=Color.GREEN, render_action=True)
            agent.pos_rew = torch.zeros(batch_dim, device=world.device)
            agent.collision_rew = agent.pos_rew.clone()
            agent.goal = goal
            world.add_agent(agent)
        world._finalize(self.scenario_id)
        self.pos_rew = torch.zeros(batch_dim, device=world.device)
        self.final_rew = self.pos_rew.clone()
        # (previous_distance_to_goal, previous_distance_to_agents) of every agent: f32[B, N, 2] in HBM
        self.shaping = torch.zeros(batch_dim, self.n_agents, 2, dtype=torch.float32, device=world.compute_device)
        return world

    def _spec(self) -> "_lib.SwarmRewardSpec":
        w = self.world
        w._sync_constants()
        return ops.reward_spec(_lib.REWARD_FLOCKING, w.batch_dim, self.n_agents, goal_x=w.cfg.goal_x, goal_y=w.cfg.goal_y,
                               goal_radius=w.landmarks[0].shape.radius, agent_radius=w.cfg.agent_radius,
                               pos_shaping=self.pos_shaping_factor, dist_shaping=self.dist_shaping_factor,
                               desired_distance=self.desired_distance,
                               min_collision_distance=self.min_collision_distance,
                               collision_reward=float(self.agent_collision_reward))

    def set_start_centers(self, centers: Optional[torch.Tensor]) -> None:
        """Batched extension: explicit per-env start centres f32[B,2] for the next resets."""
        self._explicit_centers = centers

    def reset_world_at(self, env_index: Optional[int] = None) -> None:
        w = self.world
        w.landmarks[0].set_pos(torch.tensor([-0.8, 0.8]), None)                              # flocking:96
        if self._explicit_centers is not None:
            centers = self._explicit_centers if env_index is None else self._explicit_centers[env_index:env_index + 1]
        else:
            n = w.batch_dim if (self.per_env_centers and env_index is None) else 1
            position_range = torch.tensor([-1, 1])                                           # flocking:94
            if n == 1:
                centers = position_range + torch.normal(mean=torch.tensor([-0.6, 0.6]), std=torch.tensor([0.4, 0.4]))
            else:
                centers = position_range + torch.normal(mean=torch.tensor([-0.6, 0.6]).expand(n, 2),
                                                        std=torch.tensor([0.4, 0.4]).expand(n, 2))
            # generate_grid draws two unused deviates per grid point (flocking:70-71); draw them too so that seeded
            # runs leave the global generator where the reference leaves it
            for _ in range(2 * self.n_agents):
                torch.normal(mean=torch.tensor([0.0]), std=torch.tensor([0.1]))
        w.reset_to_grid(centers, env_index)
        # previous_distance_to_goal / previous_distance_to_agents as reset_world_at leaves them (flocking:101-121)
        ops.scenario_reward(self._spec(), w.state, self.shaping, reset=True, env_index=env_index)

    def reward(self, agent: Agent) -> torch.Tensor:
        if agent is self.world.agents[0]:                                                    # flocking:125
            w = self.world
            self.collective_reward, terms = ops.scenario_reward(self._spec(), w.state, self.shaping, want_terms=True)
            radius = w.landmarks[0].shape.radius
            for a in w.agents:
                a.pos_rew = terms[:, a.index, 0]
                a.collision_rew = terms[:, a.index, 1]
                a.dist_rew = terms[:, a.index, 2]
                a.distance_to_goal = terms[:, a.index, 3]
                a.on_goal = a.distance_to_goal < radius
        return self.collective_reward

    @property
    def previous_distance_to_goal(self) -> torch.Tensor:
        return self.shaping[:, :, 0]

    @property
    def previous_distance_to_agents(self) -> torch.Tensor:
        return self.shaping[:, :, 1]

    def observation(self, agent: Agent) -> torch.Tensor:
        """cat[pos, vel, goal] f32[B,6] (flocking:173-182)."""
        return self.world.last["obs"][:, agent.index]

    def distance_to_goal_all(self) -> torch.Tensor:
        """f32[B,N] (flocking:184-191)."""
        w = self.world
        goal = w.landmarks[0].state.pos.unsqueeze(1)
        return torch.linalg.vector_norm(w.state[:, :, 0:2] - goal, dim=-1)

    def info(self, agent: Agent) -> Dict[str, torch.Tensor]:
        return {"pos_rew": agent.pos_rew, "final_rew": self.final_rew}


class CohesionScenario(BaseScenario):
    """src/scenarios/cohesion_scenario.py:7-101: no landmark, up to nine agents on a fixed start table, observation
    cat[pos, vel] (4 floats), per-agent reward from the smallest / largest surface distance to the other agents
    (``swarm_scenario_reward``, one launch per tick for all agents and envs).  Stepped by ``swarm_sim_step`` like GoTo.
    The reference takes the min / max over everything ``torch.cat`` returns, i.e. it assumes one env; here the min / max
    are per env.  The Q-network kernels are specialised for 6-float observations, so this scenario is served at the
    environment level (world step + reward), not by the fused rollout.  Its reset keeps the reference's nine-agent start
    table (and its IndexError beyond nine agents); for larger swarms, up to 4 096 agents, the Cohesion reward is reached
    through ``ops.scenario_reward`` and ``ops.rollout_stack`` with a ``REWARD_COHESION`` spec on a state the caller
    places."""

    scenario_id = _lib.SCENARIO_GOTO
    _START = [[-1.0, -1.0], [0.0, -1.0], [0.0, 1.0], [0.0, 0.0], [1.0, 1.0], [1.0, -1.0], [-1.0, 1.0], [1.0, 0.0],
              [-1.0, 0.0]]                                                                   # cohesion:46-56

    def make_world(self, batch_dim: int, device, **kwargs) -> World:
        self.pos_shaping_factor = kwargs.get("pos_shaping_factor", 10.0)
        self.dist_shaping_factor = kwargs.get("dist_shaping_factor", 10.0)
        self.agent_radius = kwargs.get("agent_radius", 0.1)
        self.n_agents = kwargs.get("n_agents", 1)
        self.min_distance_between_entities = self.agent_radius * 2 + 0.05
        self.world_semidim = 1
        self.agent_collision_reward = -1
        self.desired_distance = 0.15
        self.min_collision_distance = 0.005
        self.collective_reward = 0
        self.sigma = 0.15
        world = World(batch_dim, device)
        for i in range(self.n_agents):
            agent = Agent(name=f"agent{i}", collide=True, color=Color.GREEN, render_action=True)
            agent.pos_rew = torch.zeros(batch_dim, device=world.device)
            agent.collision_rew = agent.pos_rew.clone()
            world.add_agent(agent)
        world._finalize(self.scenario_id)
        self.pos_rew = torch.zeros(batch_dim, device=world.device)
        self.final_rew = self.pos_rew.clone()
        self._rewards: Optional[torch.Tensor] = None
        self._rewards_version = -1
        return world

    def reset_world_at(self, env_index: Optional[int] = None) -> None:
        table = torch.tensor(self._START, dtype=torch.float32)
        for i, agent in enumerate(self.world.agents):
            agent.set_pos(table[i], batch_index=env_index)       # IndexError beyond nine agents, as in the reference

    def all_rewards(self) -> torch.Tensor:
        """f32[B,N] for the current state (cached until the world steps or resets)."""
        w = self.world
        if self._rewards is None or self._rewards_version != w.version:
            spec = ops.reward_spec(_lib.REWARD_COHESION, w.batch_dim, self.n_agents, agent_radius=w.cfg.agent_radius,
                                   sigma=self.sigma)
            self._rewards = ops.scenario_reward(spec, w.state)
            self._rewards_version = w.version
        return self._rewards

    def reward(self, agent: Agent) -> torch.Tensor:
        return self.all_rewards()[:, agent.index]

    def observation(self, agent: Agent) -> torch.Tensor:
        """cat[pos, vel] f32[B,4] (cohesion:87-94)."""
        return self.world.state[:, agent.index].clone()

    def info(self, agent: Agent) -> Dict[str, torch.Tensor]:
        return {"pos_rew": agent.pos_rew, "final_rew": self.final_rew}
