"""Kilobot classes -- same names, constants and constructor signatures as
gym_kilobots/lib/kilobot.py.  The controllers themselves (Kilobot.step :86-127, _loop :318-333,
SimplePhototaxisKilobot.step :191-203, SimpleVelocityControlKilobot.step :253-258,
SimpleAccelerationControlKilobot.step :294-300) run inside the CUDA step kernel
(csrc/kb_env.cuh: senseControl); these classes record which controller a body uses and expose the
controller state the env mirrors back from the device.
"""
import numpy as np

from .. import _abi as abi
from .. import scene as S
from ..spaces import Box
from .body import Circle


class Kilobot(Circle):
    _radius = S.KILOBOT_RADIUS

    _leg_front = np.array([.0, _radius])
    _leg_left = np.array([-0.013, -.009])
    _leg_right = np.array([+0.013, -.009])
    _light_sensor = np.array([.0, -_radius + .001])
    _led = np.array([.011, .01])

    _max_linear_velocity = S.KILOBOT_MAX_LINEAR_VELOCITY   # meters / s
    _max_angular_velocity = S.KILOBOT_MAX_ANGULAR_VELOCITY  # radians / s

    _density = S.KILOBOT_DENSITY
    _friction = S.KILOBOT_FRICTION
    _restitution = S.KILOBOT_RESTITUTION

    _linear_damping = S.LINEAR_DAMPING
    _angular_damping = S.ANGULAR_DAMPING

    _kind = None  # abstract: the reference's Kilobot._loop raises NotImplementedError (lib/kilobot.py:168)

    def __init__(self, world, position=None, orientation=None, light=None):
        if self._kind is None:
            raise NotImplementedError('Kilobot subclass needs to implement _loop')
        super().__init__(world=world, position=position, orientation=orientation, radius=self._radius)
        self._body_color = (150, 150, 150)
        self._highlight_color = (255, 255, 255)
        self._light = light
        self._ctrl = np.zeros(4)   # controller state mirrored from the device after each step
        self._setup()

    def _setup(self):
        pass

    def light_sensor_pos(self):
        return self.get_world_point((0.0, -self._radius))

    def set_color(self, color):
        self._highlight_color = color


class PhototaxisKilobot(Kilobot):
    _kind = abi.KB_KILOBOT_PHOTOTAXIS

    def _setup(self):
        self._ctrl = np.array([-np.inf, 0.0, 0.0, 0.0])  # threshold, turn direction (0 left), counters

    @property
    def turn_direction(self):
        return 'right' if self._ctrl[1] else 'left'


class SimplePhototaxisKilobot(Kilobot):
    _kind = abi.KB_KILOBOT_SIMPLE_PHOTOTAXIS

    def light_sensor_pos(self):
        return self.get_position()


class SimpleVelocityControlKilobot(Kilobot):
    _density = 2.0
    _kind = abi.KB_KILOBOT_VELOCITY

    action_space = Box(np.array([.0, -Kilobot._max_angular_velocity]),
                       np.array([Kilobot._max_linear_velocity, Kilobot._max_angular_velocity]), dtype=np.float64)
    state_space = Box(np.array([-np.inf, -np.inf, -np.inf]), np.array([np.inf, np.inf, np.inf]), dtype=np.float64)

    def __init__(self, world, *, velocity=None, **kwargs):
        super().__init__(world=world, light=None, **kwargs)
        if velocity:
            self._velocity = np.asarray(velocity, dtype=np.float64)
        else:  # lib/kilobot.py:228-229
            self._velocity = np.random.rand(2) * np.array([self._max_linear_velocity, 2 * self._max_angular_velocity])
            self._velocity[1] -= self._max_angular_velocity
        self._pending_action = None

    def set_action(self, action):
        if action is not None:
            action = np.minimum(action, self.action_space.high)
            action = np.maximum(action, self.action_space.low)
            self._velocity = action
        else:
            self._velocity = np.array([.0, .0])

    def get_action(self):
        return self._velocity

    def set_color(self, color):
        self._body_color = color


class SimpleAccelerationControlKilobot(SimpleVelocityControlKilobot):
    _density = 2.0
    _kind = abi.KB_KILOBOT_ACCELERATION

    action_space = Box(np.array([-.005, -.2 * np.pi]), np.array([.005, .2 * np.pi]), dtype=np.float64)
    state_space = Box(np.array([-np.inf, -np.inf, -np.inf, .0, -Kilobot._max_angular_velocity]),
                      np.array([np.inf, np.inf, np.inf, Kilobot._max_linear_velocity, Kilobot._max_angular_velocity]),
                      dtype=np.float64)

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self._acceleration = np.array([.0, .0])

    def get_state(self):
        pose = super(SimpleAccelerationControlKilobot, self).get_state()
        return pose + tuple(self._velocity)

    def set_action(self, action):
        if action is not None:
            action = np.minimum(action, self.action_space.high)
            action = np.maximum(action, self.action_space.low)
            self._acceleration = action
        else:
            self._acceleration = np.array([.0, .0])

    def get_action(self):
        return self._acceleration
