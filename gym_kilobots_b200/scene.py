"""Scene templates: what `KilobotsEnv._configure_environment` builds, minus the poses.

The reference's constructors (gym_kilobots/lib/body.py, lib/kilobot.py, lib/light.py) create Box2D
objects immediately; here they only record a `BodySpec` / `LightSpec`.  A `SceneSpec` is the
immutable template (shapes, materials, controller kinds, light model, simulation constants) that
is uploaded once per batch through `KbSceneDesc` (include/kb_b200.h); per-env poses travel
separately as tensors.
"""
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _abi as abi

WORLD_SCALE = 25.0  # lib/body.py:7

# lib/body.py:11-16
OBJECT_DENSITY = 2.0
OBJECT_FRICTION = 0.01
OBJECT_RESTITUTION = 0.0
LINEAR_DAMPING = 0.8
ANGULAR_DAMPING = 0.8
# lib/kilobot.py:9,25-30
KILOBOT_RADIUS = 0.0165
KILOBOT_DENSITY = 1.0
KILOBOT_FRICTION = 0.0
KILOBOT_RESTITUTION = 0.0
KILOBOT_MAX_LINEAR_VELOCITY = 0.01
KILOBOT_MAX_ANGULAR_VELOCITY = 0.5 * np.pi


@dataclass
class FixtureSpec:
    shape: int
    density: float
    friction: float
    restitution: float
    radius: float = 0.0          # circle, b2 units
    hx: float = 0.0              # box half extents, b2 units
    hy: float = 0.0
    vertices: Optional[np.ndarray] = None  # polygon input vertices [V,2], b2 units (float64 before the f32 cast)


@dataclass
class BodySpec:
    kind: int
    fixtures: List[FixtureSpec]
    linear_damping: float = LINEAR_DAMPING
    angular_damping: float = ANGULAR_DAMPING


@dataclass
class LightSpec:
    type: int
    radius: float = 0.2
    bounds: Tuple[Sequence[float], Sequence[float]] = ((-np.inf, -np.inf), (np.inf, np.inf))
    action_bounds: Tuple[Sequence[float], Sequence[float]] = ((-0.01, -0.01), (0.01, 0.01))
    relative_actions: bool = True
    max_velocity: float = np.inf

    @property
    def state_dim(self):
        return {abi.KB_LIGHT_CIRCULAR: 2, abi.KB_LIGHT_MOMENTUM: 4, abi.KB_LIGHT_LINEAR: 1}[self.type]

    @property
    def action_dim(self):
        return 1 if self.type == abi.KB_LIGHT_LINEAR else 2


@dataclass
class TaskSpec:
    """Task layer (an extension; the reference's reward hooks are abstract, kilobots_env.py:123-131).

    reward = w_position * (d0 - d1) + w_orientation * (a0 - a1) - step_penalty (+ success_bonus), where d / a are
    the distance / absolute angle between the subject (object `object`, or the swarm's mean position) and the
    per-env target before and after the env-step; done on success or after max_episode_steps."""
    mode: int = abi.KB_TASK_OBJECT_TO_TARGET
    object: int = 0
    max_episode_steps: int = 0
    w_position: float = 1.0
    w_orientation: float = 0.0
    step_penalty: float = 0.0
    success_bonus: float = 0.0
    position_tolerance: float = 0.0
    orientation_tolerance: float = np.inf

    def to_def(self):
        t = abi.KbTaskDef()
        t.mode, t.object, t.max_episode_steps = int(self.mode), int(self.object), int(self.max_episode_steps)
        t.w_position, t.w_orientation = float(self.w_position), float(self.w_orientation)
        t.step_penalty, t.success_bonus = float(self.step_penalty), float(self.success_bonus)
        t.position_tolerance, t.orientation_tolerance = float(self.position_tolerance), float(self.orientation_tolerance)
        return t


@dataclass(frozen=True)
class LocalObsSpec:
    """Per-kilobot local observation (include/kb_b200.h kb_local_observation): each kilobot's neighbours within `radius`
    metres (their count, then the `max_neighbours` nearest as (x, y, distance, 1) in the kilobot's frame), every object
    slot as (x, y, cos, sin, 1) in its frame, and the light (value, gradient x, y) at its sensor.  The parts follow each
    other in that order; `dim(M)` is the row width for a batch with M object slots."""
    radius: float
    max_neighbours: int = 8
    neighbours: bool = True
    objects: bool = True
    light: bool = False

    def __post_init__(self):
        if not (self.neighbours or self.objects or self.light):
            raise ValueError("LocalObsSpec: select at least one part")
        if not 1 <= int(self.max_neighbours) <= 32:
            raise ValueError("LocalObsSpec: max_neighbours must be in 1..32")
        r = float(self.radius)
        if not (0.0 < r <= float(np.finfo(np.float32).max) and np.float32(r) > 0.0):   # (NaN fails the comparison)
            raise ValueError("LocalObsSpec: radius must be finite and > 0 (metres)")

    @property
    def parts(self):
        return ((abi.KB_LOCAL_NEIGHBOURS if self.neighbours else 0) | (abi.KB_LOCAL_OBJECTS if self.objects else 0) |
                (abi.KB_LOCAL_LIGHT if self.light else 0))

    def slices(self, num_objects):
        """{'neighbours', 'objects', 'light'} -> the column slice of each selected part."""
        out, c = {}, 0
        for name, on, width in (("neighbours", self.neighbours, 1 + 4 * int(self.max_neighbours)),
                                ("objects", self.objects, 5 * int(num_objects)), ("light", self.light, 3)):
            if on:
                out[name] = slice(c, c + width)
                c += width
        return out

    def dim(self, num_objects):
        return sum(s.stop - s.start for s in self.slices(num_objects).values())

    def to_def(self):
        d = abi.KbLocalObsDef()
        d.radius, d.max_neighbours, d.parts = float(self.radius), int(self.max_neighbours), self.parts
        return d


@dataclass
class SceneSpec:
    bodies: List[BodySpec] = field(default_factory=list)   # objects first, then kilobots
    num_objects: int = 0
    lights: List[LightSpec] = field(default_factory=list)
    world_size: Tuple[float, float] = (2.0, 1.5)            # metres, kilobots_env.py:19
    wall_edges: int = 3                                     # open chain (pybox2d `vertices=`), SURVEY B.9-U2
    wall_friction: float = 0.2
    steps_per_action: int = 10                              # kilobots_env.py:28
    velocity_iterations: int = 10                           # :26
    position_iterations: int = 10                           # :27
    dt: float = 0.1                                         # 1 / sim_steps_per_second, :25,32
    damping_mode: int = 0
    enable_toi: bool = True
    enable_sleep: bool = True
    reward_const: float = 0.0

    @property
    def num_bodies(self):
        return len(self.bodies)

    @property
    def num_kilobots(self):
        return len(self.bodies) - self.num_objects

    @property
    def light_state_dim(self):
        return sum(l.state_dim for l in self.lights)

    @property
    def action_dim(self):
        return sum(l.action_dim for l in self.lights)

    def to_desc(self):
        """-> (KbSceneDesc, keepalive objects)."""
        nb = len(self.bodies)
        bodies = (abi.KbBodyDef * max(nb, 1))()
        for i, b in enumerate(self.bodies):
            bd = bodies[i]
            bd.kind = b.kind
            bd.num_fixtures = len(b.fixtures)
            if not 1 <= len(b.fixtures) <= abi.KB_MAX_FIXTURES:
                raise ValueError("a body needs 1..%d fixtures" % abi.KB_MAX_FIXTURES)
            bd.linear_damping = b.linear_damping
            bd.angular_damping = b.angular_damping
            for j, f in enumerate(b.fixtures):
                fd = bd.fixtures[j]
                fd.shape = f.shape
                fd.radius = f.radius
                fd.hx, fd.hy = f.hx, f.hy
                fd.density, fd.friction, fd.restitution = f.density, f.friction, f.restitution
                if f.shape == abi.KB_SHAPE_POLYGON:
                    v = np.asarray(f.vertices, dtype=np.float64)
                    if not 3 <= len(v) <= abi.KB_MAX_POLY_VERTS:
                        raise ValueError("polygon needs 3..%d vertices" % abi.KB_MAX_POLY_VERTS)
                    fd.vertex_count = len(v)
                    for k in range(len(v)):
                        fd.vx[k] = v[k, 0]
                        fd.vy[k] = v[k, 1]
        nl = len(self.lights)
        if nl > abi.KB_MAX_LIGHTS:
            raise ValueError("at most %d lights" % abi.KB_MAX_LIGHTS)
        lights = (abi.KbLightDef * max(nl, 1))()
        for i, l in enumerate(self.lights):
            ld = lights[i]
            ld.type = l.type
            ld.relative_actions = int(l.relative_actions)
            ld.radius = l.radius
            lo, hi = np.asarray(l.bounds[0], float).ravel(), np.asarray(l.bounds[1], float).ravel()
            alo, ahi = np.asarray(l.action_bounds[0], float).ravel(), np.asarray(l.action_bounds[1], float).ravel()
            for k in range(2):
                ld.bounds_lo[k] = lo[min(k, len(lo) - 1)]
                ld.bounds_hi[k] = hi[min(k, len(hi) - 1)]
                ld.action_lo[k] = alo[min(k, len(alo) - 1)]
                ld.action_hi[k] = ahi[min(k, len(ahi) - 1)]
            ld.max_velocity = l.max_velocity
        d = abi.KbSceneDesc()
        d.num_bodies = nb
        d.num_objects = self.num_objects
        d.bodies = bodies
        d.num_lights = nl
        d.lights = lights
        # kilobots_env.py:33-34,48-51: _world_scale * world_x_range[...] in float64, then float32
        w, hgt = self.world_size
        d.wall_x0 = WORLD_SCALE * (-w / 2)
        d.wall_x1 = WORLD_SCALE * (w / 2)
        d.wall_y0 = WORLD_SCALE * (-hgt / 2)
        d.wall_y1 = WORLD_SCALE * (hgt / 2)
        d.wall_edges = self.wall_edges
        d.wall_friction = self.wall_friction
        d.steps_per_action = self.steps_per_action
        d.velocity_iterations = self.velocity_iterations
        d.position_iterations = self.position_iterations
        d.dt = self.dt
        d.damping_mode = self.damping_mode
        d.enable_toi = int(self.enable_toi)
        d.enable_sleep = int(self.enable_sleep)
        d.reward_const = self.reward_const
        return d, (bodies, lights)


# ---------------------------------------------------------------------------- body templates
def circle_fixture(radius_m, density, friction, restitution):
    """lib/body.py:187-192: CreateCircleFixture(radius=radius * _world_scale, ...)."""
    return FixtureSpec(abi.KB_SHAPE_CIRCLE, density, friction, restitution, radius=radius_m * WORLD_SCALE)


def box_fixture(width_m, height_m, density=OBJECT_DENSITY, friction=OBJECT_FRICTION, restitution=OBJECT_RESTITUTION):
    """lib/body.py:136-142: CreatePolygonFixture(box=(w/2 * scale, h/2 * scale))."""
    return FixtureSpec(abi.KB_SHAPE_BOX, density, friction, restitution,
                       hx=width_m / 2 * WORLD_SCALE, hy=height_m / 2 * WORLD_SCALE)


def polygon_local_vertices(template, width, height):
    """Vertex normalisation of lib/body.py:226-241.

    `template` is [K sub-polygons, V, 2].  The sub-polygons are scaled so that the overall bounding
    box is width x height and shifted by the area-weighted mean of the sub-polygons' vertex means.
    Returns local vertices in metres, float64 [K, V, 2].
    """
    verts = np.array(template, dtype=np.float64)
    extent = verts.max(axis=(0, 1)) - verts.min(axis=(0, 1))
    verts = verts / extent
    verts = verts * np.array((width, height))
    shift = np.zeros(2)
    total = 0.0
    for sub in verts:
        x, y = sub[:, 0], sub[:, 1]
        a = 0.5 * np.abs(np.dot(x, np.roll(y, 1)) - np.dot(y, np.roll(x, 1)))
        total += a
        shift += sub.mean(axis=0) * a
    shift /= total
    return verts - shift


def polygon_fixtures(local_vertices_m, density=OBJECT_DENSITY, friction=OBJECT_FRICTION,
                     restitution=OBJECT_RESTITUTION):
    """lib/body.py:244-251: one b2PolygonShape(vertices=(v * _world_scale).tolist()) per sub-polygon."""
    return [FixtureSpec(abi.KB_SHAPE_POLYGON, density, friction, restitution, vertices=np.asarray(v) * WORLD_SCALE)
            for v in local_vertices_m]


# sub-polygon templates, lib/body.py:288-329
TRIANGLE_TEMPLATE = [[(-0.5, 0.0), (0.0, 0.0), (0.0, 1.0)]]
LFORM_TEMPLATE = [[(-0.05, 0.0), (0.1, 0.0), (0.1, 0.3), (-0.05, 0.3)],
                  [(0.1, 0.0), (0.1, -0.15), (-0.2, -0.15), (-0.2, 0.0)]]
TFORM_TEMPLATE = [[(0.0, 0.15), (0.2, 0.15), (0.2, -0.15), (0.0, -0.15)],
                  [(0.0, 0.05), (0.0, -0.05), (-0.2, -0.05), (-0.2, 0.05)]]
CFORM_TEMPLATE = [[(0.09, 0.15), (0.09, -0.15), (-0.01, -0.15), (-0.01, 0.15)],
                  [(-0.01, -0.15), (-0.11, -0.15), (-0.11, -0.08), (-0.01, -0.05)],
                  [(-0.01, 0.15), (-0.11, 0.15), (-0.11, 0.08), (-0.01, 0.05)]]


def kilobot_body(kind):
    density = 2.0 if kind in (abi.KB_KILOBOT_VELOCITY, abi.KB_KILOBOT_ACCELERATION) else KILOBOT_DENSITY  # kilobot.py:214,267
    return BodySpec(kind, [circle_fixture(KILOBOT_RADIUS, density, KILOBOT_FRICTION, KILOBOT_RESTITUTION)])


def quad_body(width, height):
    return BodySpec(abi.KB_BODY_OBJECT, [box_fixture(width, height)])


def circle_body(radius):
    return BodySpec(abi.KB_BODY_OBJECT, [circle_fixture(radius, OBJECT_DENSITY, OBJECT_FRICTION, OBJECT_RESTITUTION)])


def polygon_body(template, width, height):
    return BodySpec(abi.KB_BODY_OBJECT, polygon_fixtures(polygon_local_vertices(template, width, height)))
