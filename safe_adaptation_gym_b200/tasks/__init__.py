"""Task descriptors with the reference's class names and zero-argument constructors
(safe_adaptation_gym/tasks/__init__.py:1-32).

In the reference a Task instance carries mutable per-episode state and builds MuJoCo XML; here the
per-environment task state lives on the device (sag_core.cuh: TaskState) and a Task is an immutable
descriptor: a task id plus the constants the reference exposes (``obstacles``, ``placement_extents``,
class constants).  The numbers below are pinned against the reference by tests/test_api.py through
tests/golden/layouts.json.
"""
from typing import List, Tuple

import numpy as np

PLACEMENT_EXTENTS = (-2, -2, 2, 2)  # consts.py:9


class Task:
    """tasks/task.py:14-98"""
    task_id = -1
    name = "task"

    @property
    def obstacles(self) -> List[int]:
        # order: hazards, vases, gremlins, pillars (consts.py:11)
        return [4, 5, 0, 1]

    @property
    def placement_extents(self) -> Tuple[float, float, float, float]:
        return PLACEMENT_EXTENTS

    @property
    def arena_radius(self):
        return (self.placement_extents[2]) * np.sqrt(2.)

    def __repr__(self):
        return f"{type(self).__name__}()"


class GoToGoal(Task):  # tasks/go_to_goal.py
    GOAL_SIZE = 0.3
    GOAL_KEEPOUT = 0.4
    task_id = 3
    name = "go_to_goal"

    @property
    def obstacles(self):
        return [9, 10, 0, 1]


class GoToGoalDamping(GoToGoal):  # tasks/go_to_goal_damping.py
    task_id = 4
    name = "go_to_goal_damping"


class GoToGoalMotor(GoToGoal):  # tasks/go_to_goal_motor.py
    task_id = 5
    name = "go_to_goal_motor"


class GoToGoalScarce(GoToGoal):  # tasks/go_to_goal_scarce.py
    task_id = 6
    name = "go_to_goal_scarce"


class CatchGoal(GoToGoal):  # tasks/catch_goal.py
    MIN_RADIUS = 0.2
    MAX_RADIUS = 1.0
    SAMPLE_POINTS = 10
    task_id = 0
    name = "catch_goal"


class PressButtons(Task):  # tasks/press_buttons.py
    NUM_BUTTONS = 4
    BUTTONS_KEEPOUT = 0.2
    BUTTON_SIZE = 0.1
    BUTTON_TICKING_DELAY = 5
    task_id = 8
    name = "press_buttons"

    @property
    def obstacles(self):
        return [6, 8, 0, 0]


class PressButtonsScarce(PressButtons):  # tasks/press_buttons_scarce.py
    task_id = 9
    name = "press_buttons_scarce"


class Collect(PressButtons):  # tasks/collect.py (inherits PressButtons.obstacles)
    NUM_BUTTONS = 6
    task_id = 1
    name = "collect"

    @property
    def placement_extents(self):
        return [-2.25, -2.25, 2.25, 2.25]


class PushBox(GoToGoal):  # tasks/push_box.py
    BOX_SIZE = 0.2
    BOX_KEEPOUT = 0.5
    BOX_DENSITY = 0.001
    task_id = 10
    name = "push_box"

    @property
    def obstacles(self):
        return [2, 3, 0, 1]

    @property
    def placement_extents(self):
        return [-1.75, -1.75, 1.75, 1.75]


class PushBoxScarce(PushBox):  # tasks/push_box_scarce.py
    task_id = 11
    name = "push_box_scarce"


class HaulBox(PushBox):  # tasks/haul_box.py
    task_id = 7
    name = "haul_box"


class RollRod(PushBox):  # tasks/roll_rod.py
    ROD_LENGTH = 0.3
    ROD_RADIUS = 0.08
    BOX_KEEPOUT = 0.7
    BOX_SIZE = 0.25
    task_id = 12
    name = "roll_rod"

    @property
    def placement_extents(self):
        return -1.75, -1.75, 1.75, 1.75


class DribbleBall(PushBox):  # tasks/dribble_ball.py
    SPHERE_RADIUS = 0.14
    BOX_KEEPOUT = 0.2
    BOX_SIZE = SPHERE_RADIUS
    task_id = 2
    name = "dribble_ball"

    @property
    def placement_extents(self):
        return -1.75, -1.75, 1.75, 1.75


class Unsupervised(Task):  # tasks/unsupervised.py
    task_id = 13
    name = "unsupervised"

    @property
    def obstacles(self):
        return [5, 6, 0, 1]


__all__ = [
    "GoToGoal", "PushBox", "PressButtons", "RollRod", "DribbleBall", "Collect", "HaulBox", "CatchGoal",
    "Unsupervised", "GoToGoalScarce", "PressButtonsScarce", "PushBoxScarce", "GoToGoalDamping", "GoToGoalMotor",
]

# tasks the device path does not simulate (none: all 14 registry tasks run; kept for callers that filter on it)
DEVICE_UNSUPPORTED = frozenset()

# every concrete task class (task_id = index in the registry's alphabetical order, benchmark/__init__.py:16-20)
TASK_CLASSES = tuple(sorted((globals()[n] for n in __all__), key=lambda c: c.task_id))

# what a user-defined task may override: the two properties the device path takes from it, and what Python puts in
# every class body
_OVERRIDABLE = frozenset(("obstacles", "placement_extents"))
_CLASS_BOOKKEEPING = frozenset(("__module__", "__qualname__", "__doc__", "__dict__", "__weakref__", "__annotations__",
                                "__firstlineno__", "__static_attributes__", "__orig_bases__", "__parameters__"))


def registry_base(task: Task) -> type:
    """The registry class a task instance derives from (the first of TASK_CLASSES in its MRO)."""
    for cls in type(task).__mro__:
        if cls in TASK_CLASSES:
            return cls
    raise TypeError(f'{type(task).__name__} does not derive from a registry task ({", ".join(__all__)})')


def definition(task: Task):
    """A task as the device path sees it: (base class, obstacles [4 ints], placement_extents [4 floats]).

    Only ``obstacles`` and ``placement_extents`` may differ from the base; a subclass that overrides anything else
    (class constants such as ``GOAL_SIZE``, methods such as a reward, other attributes) raises NotImplementedError
    naming it."""
    base = registry_base(task)
    for cls in type(task).__mro__:
        if cls is base:
            break
        for name in cls.__dict__:
            if name not in _OVERRIDABLE and name not in _CLASS_BOOKKEEPING:
                raise NotImplementedError(f'{type(task).__name__} overrides {name!r}: the device path runs '
                                          f'{base.__name__} with its own obstacles and placement_extents only')
    for name in vars(task):
        raise NotImplementedError(f'{type(task).__name__} sets the instance attribute {name!r}: the device path runs '
                                  f'{base.__name__} with its own obstacles and placement_extents only')
    obstacles = [int(v) for v in task.obstacles]
    extents = [float(v) for v in task.placement_extents]
    if len(obstacles) != 4 or len(extents) != 4:
        raise ValueError(f'{type(task).__name__}: obstacles and placement_extents need 4 entries each')
    return base, obstacles, extents


def is_registry_equivalent(task: Task) -> bool:
    """Whether a task runs exactly as its registry base (the same obstacles and extents, nothing else overridden)."""
    base, obstacles, extents = definition(task)
    b = base()
    return obstacles == [int(v) for v in b.obstacles] and extents == [float(v) for v in b.placement_extents]
