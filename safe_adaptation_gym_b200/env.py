"""Batched drop-in variant of ``SafeAdaptationGym`` (reference: safe_adaptation_gym/safe_adaptation_gym.py:21-257).

Same method names and argument meaning as the reference env, with a leading batch dimension:

    obs[N, D], reward[N], done[N], info{'cost'[N], 'bound'[N]} = env.step(actions[N, nu])
    obs[N, D] = env.reset(options={'task': task_or_list_of_tasks})

Returned tensors are fresh copies by default, like the arrays the reference returns; ``copy_outputs=False`` hands out the
internal output buffers instead (valid until the next call -- the zero-copy mode for throughput loops).
With ``max_episode_steps > 0`` the env auto-resets like a vectorised gym wrapper: an environment whose episode ended
(time limit, or done after a physics error) is reset inside ``step``; its row of ``obs`` is the FIRST observation of the
new episode, ``done`` is True for it and ``info['truncated']`` marks the time-limit endings.

``step`` (both output modes, with or without auto-reset), ``rollout``, ``observation``, ``copy_envs`` and
``evaluate_actions`` (with device tensors) may be recorded in a CUDA graph
(``torch.cuda.graph``), together with the policy that computes the actions; every replay behaves like issuing the same
calls again.  ``seed``, ``set_task`` and ``load_state_dict`` between replays are seen by the graph, except that a
``set_task`` which changes whether any environment runs ``Unsupervised`` changes the reward buffer ``step`` records:
capture again after it.  No Python runs during a replay, so errors recorded by replayed steps are raised by
``check_errors()``.  The methods that synchronise raise ``RuntimeError`` while a capture is open.

Task switches per environment: ``set_next_task`` queues a task for each environment's NEXT reset (the auto-reset inside
``step``, ``reset``, ``reset_envs``), so that every environment of a staggered batch moves on to its next task when its
own episode ends, without cutting any running episode short.  At that reset the environment's finished episode and
statistics stay with the old task (``task_stats``), and it starts a fresh Task instance of the queued task (new
ctrl-range scale and bound draws).  With a device tensor of ids it may be recorded in a CUDA graph with the policy and
``step``, so a graphed adaptation loop can walk through tasks; ``task_ids`` tells which task each environment runs now.
``set_task(task, mask)`` switches the masked environments at once (their running episodes are cut short and not counted).

User-defined tasks: an instance of a subclass of a registry task that overrides ``obstacles`` and / or
``placement_extents`` runs the base's logic with its own obstacle counts and extents, under a task id of its own (14,
15, ... per batch; ``task_id_of``).  Everything that takes a task takes one.  Defining the first one switches the batch
to another kernel set: a CUDA graph captured before it must be captured again.

All per-step arithmetic (dynamics, reward / goal logic, cost, pseudo-lidar) runs in the CUDA library behind
the C ABI of ``include/sag_b200.h``; this class only owns torch tensors and passes raw pointers.  There is
no CPU fallback: without the built library and a CUDA device construction raises.
"""
import ctypes as C
from typing import Dict, Optional, Sequence, Union

import numpy as np
import torch

from safe_adaptation_gym_b200 import _abi
from safe_adaptation_gym_b200 import tasks as _tasks
from safe_adaptation_gym_b200.spaces import Box
from safe_adaptation_gym_b200.utils import ResamplingError

# World.DEFAULT, world.py:17-34
WORLD_DEFAULT = {
    'placements_margin': 0.0, 'robot_keepout': 0.4, 'hazards_size': 0.2, 'vases_size': 0.1, 'pillars_size': 0.2,
    'gremlins_size': 0.1, 'hazards_keepout': 0.18, 'gremlins_keepout': 0.4, 'vases_keepout': 0.15,
    'pillars_keepout': 0.3, 'gremlins_travel': 0.35, 'obstacles_size_noise_scale': 0.0,
    'robot_ctrl_range_scale': 0.0, 'action_noise': 0.01, 'max_bound': 25, 'random_bound': False,
}
# max_layout_draws: draw budget of a layout; num_gremlins: Task.obstacles[2] of a user-defined task (task.py:70; every
# task of the reference's registry has 0 gremlins) -- gremlins per environment, world.py:157-165
_EXTRA_KEYS = {'max_layout_draws', 'num_gremlins'}
_ROBOT_TO_CONTROL_FREQUENCY = {'doggo': 12, 'point': 5, 'car': 10}  # safe_adaptation_gym.py:15-19


def _capturing() -> bool:
    """True while the current CUDA stream is recording a graph."""
    try:
        return torch.cuda.is_current_stream_capturing()
    except RuntimeError:  # no usable CUDA driver: nothing can be recording
        return False


def _robot_name(path: str) -> str:
    base = path.replace('\\', '/').split('/')[-1]
    return base[:-4] if base.endswith('.xml') else base


class BatchedSafeAdaptationGym:
    NUM_LIDAR_BINS = 16
    LIDAR_MAX_DIST = 5.
    BASE_SENSORS = ['accelerometer', 'velocimeter', 'gyro', 'magnetometer']

    def __init__(self,
                 robot_base: str,
                 rgb_observation: bool = False,
                 config: Optional[Dict] = None,
                 render_lidars_and_collision: bool = False,
                 render_options: Optional[Dict] = None,
                 num_envs: int = 1,
                 device: Union[str, torch.device, None] = None,
                 env_id_base: int = 0,
                 max_episode_steps: int = 0,
                 copy_outputs: bool = True,
                 _test_lib=None):
        if rgb_observation:
            raise NotImplementedError('rgb_observation needs a rasteriser and is outside the B200 hot path '
                                      '(reference: safe_adaptation_gym.py:122-126)')
        self.robot_name = _robot_name(robot_base)
        if self.robot_name not in _ROBOT_TO_CONTROL_FREQUENCY:
            raise KeyError(self.robot_name)
        if self.robot_name not in ('point', 'car'):
            raise NotImplementedError(f"robot '{self.robot_name}' is not implemented on the device path (3-D articulated body)")
        cfg = dict(WORLD_DEFAULT)
        for k, v in (config or {}).items():
            if k not in WORLD_DEFAULT and k not in _EXTRA_KEYS:
                raise KeyError(f'unknown config key {k!r}')
            cfg[k] = v
        self.base_config = cfg
        self.num_envs = int(num_envs)
        if _test_lib is None:
            self._lib = _abi.load()
            if not torch.cuda.is_available():
                raise _abi.SagError('no CUDA device: the B200 path has no CPU fallback')
            self.device = torch.device(device if device is not None else 'cuda:0')
            if self.device.type != 'cuda':
                raise _abi.SagError('the B200 path runs on CUDA devices only')
            dev_index = self.device.index or 0
        else:  # tests/hostemu: same ABI compiled for the host, CPU tensors
            self._lib = _test_lib
            self.device = torch.device('cpu')
            dev_index = 0
        L = self._lib
        c = L.default_config()
        c.n_envs = self.num_envs
        c.robot = 1 if self.robot_name == 'car' else 0
        c.env_id_base = int(env_id_base)
        c.max_episode_steps = int(max_episode_steps)
        c.max_layout_draws = int(cfg.get('max_layout_draws', 0))
        c.random_bound = 1 if cfg['random_bound'] else 0
        c.num_gremlins = int(cfg.get('num_gremlins', 0))
        for k in ('placements_margin', 'robot_keepout', 'hazards_size', 'vases_size', 'pillars_size', 'gremlins_size',
                  'hazards_keepout', 'gremlins_keepout', 'vases_keepout', 'pillars_keepout', 'gremlins_travel',
                  'robot_ctrl_range_scale', 'action_noise', 'max_bound'):
            setattr(c, k, float(cfg[k]))
        self._seed = int(np.random.randint(2**32))  # safe_adaptation_gym.py:47
        c.seed = self._seed
        self._h = C.c_void_p()
        L.check(L.L.sag_create(C.byref(c), dev_index, C.byref(self._h)))
        self.stride = L.L.sag_stride(self._h)
        self.obs_dim = L.L.sag_obs_dim(self._h)
        self.max_episode_steps = int(max_episode_steps)
        self.env_id_base = int(env_id_base)
        self.copy_outputs = bool(copy_outputs)
        n, dev = self.num_envs, self.device
        self._obs = torch.empty((n, self.obs_dim), dtype=torch.float32, device=dev)
        self._reward = torch.empty((n,), dtype=torch.float64, device=dev)
        self._reward2 = torch.empty((n, 2), dtype=torch.float64, device=dev)
        self._cost = torch.empty((n,), dtype=torch.uint8, device=dev)
        self._done = torch.empty((n,), dtype=torch.uint8, device=dev)
        self._was_reset = torch.zeros((n,), dtype=torch.uint8, device=dev)
        self._eval_cost = torch.empty((n,), dtype=torch.float64, device=dev)     # evaluate_actions (copy_outputs=False)
        self._eval_length = torch.empty((n,), dtype=torch.int32, device=dev)
        self._bound = torch.full((n,), float(cfg['max_bound']), dtype=torch.float64, device=dev)
        self._task_ids = None
        self._tasks = None
        self._any_unsupervised = False
        self._custom = []          # user-defined tasks of this batch, in order of definition: id = NUM_TASKS + index
        self._next_armed = False   # set_next_task has been called: step refreshes a random bound after the auto-reset
        self._action_space = Box(-1, 1, (2,), dtype=np.float32)  # safe_adaptation_gym.py:49-50 (nu = 2)
        self._observation_space = None

    # ------------------------------------------------------------------------------------------
    def __del__(self):
        try:
            if getattr(self, '_h', None):
                self._lib.L.sag_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def close(self):
        self.__del__()

    def _stream(self):
        if self.device.type == 'cuda':
            return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        return C.c_void_p(0)

    @staticmethod
    def _p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else None

    # ------------------------------------------------------------------------------------------
    # reference API
    # ------------------------------------------------------------------------------------------
    def _out(self, t):
        return t.clone() if self.copy_outputs else t

    @staticmethod
    def _forbid_capture(what: str):
        if _capturing():
            raise RuntimeError(f'{what} synchronises with the device and cannot be recorded in a CUDA graph; '
                               'call it outside the capture (a graph replayed afterwards sees its effect)')

    def _raise_recorded_errors(self, where: str):
        """The reference raises out of the call in which the condition occurs; the kernels record it in mapped host
        memory instead, which is read here WITHOUT synchronising -- so an error of a step that is still in flight is
        raised by the next call (or by check_errors(), which synchronises)."""
        w = self._lib.L.sag_error_flags(self._h, 1)
        if w & _abi.FLAG_RESAMPLE_FAILED:
            raise ResamplingError('Failed to generate goal' if where == 'step' else 'Failed to generate layout')  # go_to_goal.py:80 / world.py:189
        if w & _abi.ERR_BAD_TASK_ID:
            raise ValueError('task id out of range')
        if w & _abi.ERR_BAD_ENV_INDEX:
            raise IndexError('copy_envs: a source index was out of range or named an environment the same call '
                             'overwrites; those pairs were not applied')

    def step(self, action):
        """safe_adaptation_gym.py:56-83.  `action`: [N, 2] tensor / array in [-1, 1].

        May be recorded in a CUDA graph (``torch.cuda.graph``) with the action already a tensor on this env's device;
        a host / numpy action raises ``RuntimeError`` under capture.  A replay runs no Python: conditions the replayed
        steps record (a goal that could not be sampled) are raised by ``check_errors()``, which a graphed loop should
        call at the points where it wants them surfaced.  The tensors returned during the capture are the ones every
        replay rewrites.
        """
        act = self._as_action(action)
        L = self._lib
        r2 = self._reward2 if self._any_unsupervised else None
        L.check(L.L.sag_step(self._h, self._p(act), self._p(self._obs), self._p(self._reward), self._p(r2),
                             self._p(self._cost), self._p(self._done), self._stream()))
        reward = self._reward2 if self._any_unsupervised else self._reward
        was_reset = None
        if self.max_episode_steps > 0:
            # auto-reset: the kernel resets the flagged environments, writes the first observation of their new episode
            # into their rows and reports which ones it reset
            L.check(L.L.sag_reset_obs(self._h, None, 1, 0, self._p(self._obs), self._p(self._was_reset), self._stream()))
            was_reset = self._was_reset.to(torch.bool)
            if self._next_armed and self.base_config['random_bound']:
                # an environment that switched task drew a new bound (world.py:75-78); in place: a graph may export it
                L.check(L.L.sag_bound(self._h, self._p(self._bound), self._stream()))
        if self.copy_outputs:
            # fresh arrays, as the reference returns them (safe_adaptation_gym.py:80-83) -- one launch for all of them
            n, dev = self.num_envs, self.device
            obs = torch.empty((n, self.obs_dim), dtype=torch.float32, device=dev)
            rew = torch.empty_like(reward)
            cost = torch.empty((n,), dtype=torch.float32, device=dev)
            done = torch.empty((n,), dtype=torch.bool, device=dev)
            bound = torch.empty((n,), dtype=torch.float64, device=dev)
            L.check(L.L.sag_export_outputs(self._h, self._p(self._obs), self._p(reward), 2 if self._any_unsupervised else 1,
                                           self._p(self._cost), self._p(self._done), self._p(self._bound), self._p(obs), self._p(rew),
                                           self._p(cost), self._p(done), self._p(bound), self._stream()))
        else:  # views of the internal buffers, valid until the next call
            obs, rew, bound = self._obs, reward, self._bound
            cost, done = self._cost.to(torch.float32), self._done.view(torch.bool)
        info = {'cost': cost, 'bound': bound}
        if was_reset is not None:
            info['truncated'] = was_reset & ~done   # ended by the time limit, not by a physics error
            done = done | was_reset
        self._raise_recorded_errors('step')
        return obs, rew, done, info

    def evaluate_actions(self, actions, discount: float = 1.0):
        """Run a horizon of actions and return what a planner scores a candidate by: ``obs, ret, cost, length``.

        `actions`: float32 tensor [H, N, 2] on this env's device, H >= 1.  Every environment takes exactly H steps with
        ``actions[h]``; afterwards its state (every ``_FIELDS`` field, ``task_stats``, the Philox draw counters) is
        bit-identical to what H calls of ``step(actions[h])`` leave.  With weights ``w_0 = 1``, ``w_{h+1} = w_h *
        discount`` (float64, formed left to right) and ``L_e = min(H, 1 + the first h at which step h reported
        done[e])`` (a physics error):

        - ``obs``: float32 [N, obs_dim], the observation of the last step, bit-identical to the H-th ``step``'s;
        - ``ret``: float64 [N] (or [N, 2] when this batch records Unsupervised's reward pair, as ``step``),
          ``sum_{h < L_e} w_h * r_h[e]``, each product rounded and then added, in step order from zero;
        - ``cost``: float64 [N], the same sum over the binary step cost;
        - ``length``: int32 [N], ``L_e``.

        With ``discount=1.0`` the sums equal those of a loop ``ret += r; cost += info['cost']`` over H ``step`` calls,
        stopped at each environment's first done.  Steps after ``L_e`` still run but do not count.  Only the last step
        builds an observation, so a horizon costs less than H steps.  Outputs follow ``copy_outputs`` like ``step``.

        A batch with ``max_episode_steps > 0`` is refused (``ValueError``): ``step`` would auto-reset in the middle of
        the horizon.  May be recorded in a CUDA graph (with ``copy_envs`` and the policy or sampler that fills
        `actions`); H and `discount` are fixed by the capture.  Errors recorded during the call (a goal that could not
        be resampled) raise as they do for ``step``, and through ``check_errors()`` after replays."""
        if self.max_episode_steps > 0:
            raise ValueError('evaluate_actions needs a batch without a time limit (max_episode_steps = 0): step would '
                             'auto-reset environments in the middle of the horizon')
        on_device = (torch.is_tensor(actions) and actions.device.type == self.device.type
                     and (actions.device.index or 0) == (self.device.index or 0))
        if not on_device:
            if _capturing():
                raise RuntimeError('under CUDA graph capture evaluate_actions needs the actions already on the env\'s '
                                   f'device ({self.device}); a host array would record a copy from pageable memory')
            raise ValueError(f'actions must be a float32 tensor on {self.device}')
        if actions.dtype != torch.float32 or actions.dim() != 3 or tuple(actions.shape[1:]) != (self.num_envs, 2) \
                or actions.shape[0] < 1:
            raise ValueError(f'need a float32 tensor of shape (H >= 1, {self.num_envs}, 2), got {actions.dtype} '
                             f'{tuple(actions.shape)}')
        act = actions.contiguous()
        n, dev = self.num_envs, self.device
        cols = 2 if self._any_unsupervised else 1
        if self.copy_outputs:
            obs = torch.empty((n, self.obs_dim), dtype=torch.float32, device=dev)
            ret = torch.empty((n, 2) if cols == 2 else (n,), dtype=torch.float64, device=dev)
            cost = torch.empty((n,), dtype=torch.float64, device=dev)
            length = torch.empty((n,), dtype=torch.int32, device=dev)
        else:  # the internal buffers, valid until the next call
            obs, cost, length = self._obs, self._eval_cost, self._eval_length
            ret = self._reward2 if cols == 2 else self._reward
        L = self._lib
        L.check(L.L.sag_evaluate_actions(self._h, int(act.shape[0]), self._p(act), C.c_double(float(discount)),
                                         self._p(obs), self._p(ret), cols, self._p(cost), self._p(length),
                                         self._stream()))
        self._raise_recorded_errors('step')
        return obs, ret, cost, length

    def reset(self, *, seed: Optional[int] = None, return_info: bool = False, options: Optional[dict] = None):
        """safe_adaptation_gym.py:85-107"""
        self._forbid_capture('reset')
        assert self._task_ids is not None or (options is not None and 'task' in options), (
            'A task should be first set before reset.')
        if seed is not None:
            self.seed(seed)
        if options is not None and 'task' in options:
            self.set_task(options['task'])
            return self.observation
        self._reset_all(new_task=False)
        return self.observation

    def seed(self, seed=None):
        """safe_adaptation_gym.py:113-118: new stream key; episode counters restart"""
        self._forbid_capture('seed')
        self._seed = int(np.random.randint(2**32)) if seed is None else int(seed)
        self._lib.check(self._lib.L.sag_seed(self._h, C.c_uint64(self._seed)))

    def _task_list(self, task, allow_none: bool):
        """A Task, or a sequence of N Tasks (or None where `allow_none`), validated -> list of N."""
        if isinstance(task, _tasks.Task):
            task_list = [task] * self.num_envs
        else:
            task_list = list(task)
            if len(task_list) != self.num_envs:
                raise ValueError(f'need {self.num_envs} tasks, got {len(task_list)}')
        for t in task_list:
            if t is None and allow_none:
                continue
            if t.name in _tasks.DEVICE_UNSUPPORTED:
                raise NotImplementedError(f"task '{t.name}' is not implemented on the device path yet")
        return task_list

    def set_task(self, task, mask=None):
        """safe_adaptation_gym.py:165-168.  `task`: a Task, or a sequence of N Tasks (one per environment).

        Without `mask` every environment starts a fresh Task instance now, and tasks queued with ``set_next_task`` are
        dropped.  With `mask` (N booleans) only the masked environments switch now, to fresh Task instances of their
        entries of `task`; their running episodes are cut short and not counted in ``task_stats``.  The others keep
        running and keep their queued tasks.

        A CUDA graph that records ``step`` must be captured again when this changes whether any environment runs
        ``Unsupervised`` (its reward is a pair, written to another buffer)."""
        self._forbid_capture('set_task')
        task_list = self._task_list(task, allow_none=False)
        ids = torch.tensor([self.task_id_of(t) for t in task_list], dtype=torch.int32)
        if mask is not None:
            m = torch.as_tensor(mask).to(device=self.device, dtype=torch.bool).reshape(self.num_envs)
            unsup = self._is_unsupervised(ids)
            self._any_unsupervised = self._any_unsupervised or bool(unsup[m.cpu()].any())
            # the masked environments get the task queued and are reset: the reset consumes the slot
            queued = torch.where(m, ids.to(self.device), self.get_field('next_task')[:self.num_envs]).contiguous()
            self._lib.check(self._lib.L.sag_set_next_tasks(self._h, self._p(queued), self._stream()))
            self._reset_all(new_task=False, mask=m, switch=True)
            self._tasks_from_ids(self.task_ids.cpu())
            return
        self._tasks = task_list
        self._task_ids = ids.to(self.device)
        self._any_unsupervised = bool(self._is_unsupervised(ids).any())
        self._lib.check(self._lib.L.sag_set_tasks(self._h, self._p(self._task_ids), self._stream()))
        self._observation_space = None
        self._reset_all(new_task=True)

    def set_next_task(self, task):
        """Queue the task each environment takes at its NEXT reset (-1 / None = none); replaces every environment's
        queue slot.  `task`: a Task (all environments), a sequence of N Tasks or None, or an int32 tensor [N] of task
        ids on this env's device.

        The next reset of an environment with a queued task -- the auto-reset inside ``step``, ``reset``,
        ``reset_envs`` -- credits its finished episode and its statistics to the task it ran under, then starts a fresh
        Task instance of the queued task (new ctrl-range scale and bound draws, even if the id is unchanged) and clears
        the slot.  The other environments reset as before.  ``set_task`` without a mask clears every slot.

        May be recorded in a CUDA graph with a device tensor (a host sequence raises ``RuntimeError`` under capture).
        Host input is validated; a device tensor is checked where it is consumed: an id outside [-1, 14 + the number of
        user-defined tasks) is not applied
        and raises ``ValueError`` at the next call that checks errors (``step``, ``check_errors``).  Queuing
        ``Unsupervised`` into a batch whose reward is not the pair raises ``ValueError``: ``step`` would have to record
        another reward buffer, so use ``set_task`` for that.  With a device tensor this is the caller's rule.  With
        ``random_bound``, ``step`` refreshes ``info['bound']`` after the auto-reset once this has been called: capture
        a graph of ``step`` after the first call."""
        on_device = (torch.is_tensor(task) and task.device.type == self.device.type
                     and (task.device.index or 0) == (self.device.index or 0))
        if on_device:
            if task.dtype != torch.int32 or tuple(task.shape) != (self.num_envs,):
                raise ValueError(f'need an int32 tensor of shape ({self.num_envs},), got {task.dtype} {tuple(task.shape)}')
            ids = task.contiguous()
        else:
            if _capturing():
                raise RuntimeError('under CUDA graph capture set_next_task needs an int32 tensor of task ids on the env\'s '
                                   f'device ({self.device}); a host sequence would record a copy from pageable memory')
            if torch.is_tensor(task) or isinstance(task, np.ndarray):
                by_id = self._classes_by_id()
                raw = [int(i) for i in np.asarray(task.cpu() if torch.is_tensor(task) else task).reshape(-1)]
                bad = [i for i in raw if i != -1 and i not in by_id]
                if bad:
                    raise ValueError(f'task id {bad[0]} out of range [-1, {len(by_id)})')
                task = [None if i == -1 else by_id[i]() for i in raw]
            task_list = self._task_list(task, allow_none=True)
            if not self._any_unsupervised and any(isinstance(t, _tasks.Unsupervised) for t in task_list):
                raise ValueError("Unsupervised's reward is a pair, which this batch's step does not record: "
                                 'switch to it with set_task')
            ids = torch.tensor([-1 if t is None else self.task_id_of(t) for t in task_list],
                               dtype=torch.int32).to(self.device)
        self._lib.check(self._lib.L.sag_set_next_tasks(self._h, self._p(ids), self._stream()))
        self._next_armed = True

    def _copy_world(self) -> dict:
        """The configuration two batches must share for their environments to exchange states, as the library compares
        it (sag_layout.h: copy_incompatibility): a keepout counts as the larger of it and its object's size
        (world.py:60-66)."""
        c = self.base_config
        w = {'robot': self.robot_name, 'num_gremlins': int(c.get('num_gremlins', 0)), 'random_bound': bool(c['random_bound'])}
        for k in ('placements_margin', 'robot_keepout', 'gremlins_travel', 'robot_ctrl_range_scale', 'max_bound'):
            w[k] = float(c[k])
        for kind in ('hazards', 'vases', 'pillars', 'gremlins'):
            w[kind + '_size'] = float(c[kind + '_size'])
            w[kind + '_keepout (effective)'] = max(float(c[kind + '_keepout']), float(c[kind + '_size']))
        w['user-defined tasks'] = self._definitions()
        return w

    def copy_envs(self, index, source=None):
        """Give environments of this batch the complete state of environments of `source` (default: this batch).

        `index` has one entry per environment j of this batch: j takes the state of environment index[j] of `source`,
        -1 leaves j untouched.  So K copies of each of N environments of `env` into a planning batch of N*K is
        ``plan.copy_envs(torch.arange(N * K, device=dev, dtype=torch.int32) // K, source=env)``.  `index` is an int32
        tensor [num_envs] on this env's device (stream-ordered, may be recorded in a CUDA graph) or a host sequence /
        ndarray / tensor (validated here; raises ``RuntimeError`` under capture).

        What a copy carries: every state field (robot, objects, task state and id, flags, car extras, gremlins, the
        queued next task), bit for bit, with the episode number and the in-step draw counter.  What it does not: the
        Philox key and the global environment id -- the copy draws its action noise and its goal, button and radius
        resamples from THIS batch's streams.  So with the same seed and an ``env_id_base`` that gives a copy its
        source's global id, the copy replays the source exactly (through goal resamples, auto-resets and queued task
        switches); with another global id it follows the source until its first in-step draw.

        Statistics (``task_stats``): the destination's own episode is settled as a reset settles it -- one that has
        finished (time limit or done) but has not been reset yet counts under its old task, an unfinished one is dropped;
        its earlier finished episodes stay with its old task; the copied episode, with the return and cost it has gathered so far, is
        credited to this batch in full when it finishes.

        Within one batch a pair j <- s (s != j) is applied only if s is not itself overwritten by the same call
        (index[s] is -1 or s); j <- j does nothing.  Host input breaking that rule, of the wrong length or dtype raises
        ``ValueError``, an index outside [-1, source.num_envs) ``IndexError``.  On a device tensor such pairs are not
        applied and raise ``IndexError`` at the next call that checks errors (``step``, ``check_errors``).

        The two batches must be on the same device and share robot, gremlins, object sizes, keepouts, placement margins,
        gremlin travel, ctrl-range scale and the bound settings (``ValueError`` otherwise); they may differ in
        num_envs, seed, env_id_base, max_episode_steps, max_layout_draws and action_noise -- a noise-free planning
        batch without a time limit is the intended use.  A copy may bring ``Unsupervised`` (whose reward is a pair)
        into this batch only if its ``step`` already records the pair: host input checks the copied environments, a
        device tensor is refused whenever `source` records the pair and this batch does not."""
        src = self if source is None else source
        self._check_copy_source(src)
        on_device = (torch.is_tensor(index) and index.device.type == self.device.type
                     and (index.device.index or 0) == (self.device.index or 0))
        if on_device:
            if index.dtype != torch.int32 or tuple(index.shape) != (self.num_envs,):
                raise ValueError(f'need an int32 tensor of shape ({self.num_envs},), got {index.dtype} {tuple(index.shape)}')
            if src._any_unsupervised and not self._any_unsupervised:
                raise ValueError("the source batch records Unsupervised's reward pair and this batch does not: a copy "
                                 'could bring Unsupervised in (set_task it here first)')
            idx = index.contiguous()
        else:
            if _capturing():
                raise RuntimeError('under CUDA graph capture copy_envs needs an int32 tensor of indices on the env\'s '
                                   f'device ({self.device}); a host sequence would record a copy from pageable memory')
            raw = np.asarray(index.cpu() if torch.is_tensor(index) else index)
            if raw.shape != (self.num_envs,):
                raise ValueError(f'need {self.num_envs} source indices, got shape {raw.shape}')
            if raw.dtype.kind not in 'iu':
                raise ValueError(f'source indices must be integers, got {raw.dtype}')
            raw = raw.astype(np.int64)
            bad = raw[(raw < -1) | (raw >= src.num_envs)]
            if bad.size:
                raise IndexError(f'source index {int(bad[0])} out of range [-1, {src.num_envs})')
            if src is self:
                j = np.nonzero((raw >= 0) & (raw != np.arange(self.num_envs)))[0]
                t = raw[raw[j]]
                clash = (t != -1) & (t != raw[j])
                if clash.any():
                    k = int(j[clash][0])
                    raise ValueError(f'environment {k} copies environment {int(raw[k])}, which the same call overwrites')
            if not self._any_unsupervised:
                used = torch.as_tensor(raw[raw >= 0], device=src.device)
                if bool(self._is_unsupervised(src.task_ids[used]).any()
                        | self._is_unsupervised(src.get_field('next_task')[used]).any()):
                    raise ValueError("a copied environment runs or has queued Unsupervised, whose reward is a pair that "
                                     'this batch\'s step does not record: set_task it here first')
            idx = torch.as_tensor(raw, dtype=torch.int32).to(self.device)
        self._lib.check(self._lib.L.sag_copy_envs(self._h, src._h, self._p(idx), self._stream()))
        self._next_armed = self._next_armed or src._next_armed   # copies carry queued next tasks
        if self.base_config['random_bound']:
            # the copies carry their source's bound draw; in place: a CUDA graph may export it
            self._lib.check(self._lib.L.sag_bound(self._h, self._p(self._bound), self._stream()))
        if not on_device:
            self._tasks_from_ids(self.task_ids.cpu())

    def _check_copy_source(self, src):
        if not isinstance(src, BatchedSafeAdaptationGym):
            raise TypeError(f'source must be a BatchedSafeAdaptationGym, got {type(src).__name__}')
        same_device = (src.device.type, src.device.index or 0) == (self.device.type, self.device.index or 0)
        if src._lib is not self._lib or not same_device:
            raise ValueError(f'the source batch runs on another device or library ({src.device} != {self.device})')
        mine, theirs = self._copy_world(), src._copy_world()
        for k, v in mine.items():
            if theirs[k] != v:
                raise ValueError(f'the batches differ in {k}: {theirs[k]!r} != {v!r}')

    @property
    def task_ids(self) -> torch.Tensor:
        """int32 [N] on the env's device: the task each environment runs now (it changes at the resets that consume
        queued tasks).  May be read inside a CUDA graph."""
        return self.get_field('task_i32')[0, :self.num_envs]

    def _tasks_from_ids(self, ids: torch.Tensor):
        """The host-side task list from the ids the device holds (int32 [N] on the host)."""
        by_id = self._classes_by_id()
        self._tasks = [by_id[int(i)]() for i in ids.tolist()]
        self._task_ids = ids.to(self.device)

    # ---- user-defined tasks -------------------------------------------------------------------
    def task_id_of(self, task) -> int:
        """The task id of `task` on this batch, for ``set_next_task`` with a device tensor and for reading
        ``task_ids`` / ``task_stats``.  A registry task, or a subclass whose ``obstacles`` and ``placement_extents``
        equal its base's, has the registry id.  Another subclass of a registry task (a user-defined task) gets an id of
        its own, 14, 15, ... in order of first use on this batch, one per class; the first use defines it, which
        synchronises (``RuntimeError`` under CUDA graph capture).  A definition restored by ``load_state_dict`` is
        taken by the first class with the same base, obstacles and extents, so a resumed batch keeps its ids.  Raises ``NotImplementedError`` for a subclass that
        overrides anything besides ``obstacles`` and ``placement_extents`` and ``ValueError`` for a definition the
        device cannot run (see ``_check_definition``)."""
        if type(task) in _tasks.TASK_CLASSES:
            return type(task).task_id
        base, obstacles, extents = _tasks.definition(task)
        for k, c in enumerate(self._custom):
            if c['cls'] is type(task):
                return _abi.NUM_TASKS + k
        if _tasks.is_registry_equivalent(task):
            return base.task_id
        for k, c in enumerate(self._custom):
            if not c['claimed'] and (c['base'], c['obstacles'], c['extents']) == (base, obstacles, extents):
                c['cls'], c['claimed'] = type(task), True
                return _abi.NUM_TASKS + k
        return self._define(type(task), base, obstacles, extents)

    def _check_definition(self, name, base, obstacles, extents):
        if any(v < 0 for v in obstacles):
            raise ValueError(f'{name}: obstacle counts must be >= 0, got {obstacles}')
        ng = int(self.base_config.get('num_gremlins', 0))
        if obstacles[2] != ng:
            raise ValueError(f'{name}: obstacles[2] = {obstacles[2]} gremlins, but this batch runs num_gremlins = {ng} '
                             '(gremlins are a batch setting: make the batch with config={"num_gremlins": k})')
        # the base's task objects: its buttons, goal + box, or goal
        n_task = (base.NUM_BUTTONS if issubclass(base, _tasks.PressButtons) else 2 if issubclass(base, _tasks.PushBox)
                  else 1)
        if sum(obstacles) + n_task > _abi.MAX_SLOTS:
            raise ValueError(f'{name}: {sum(obstacles)} obstacles + {n_task} task objects exceed {_abi.MAX_SLOTS} slots')
        if not (extents[0] < extents[2] and extents[1] < extents[3]):
            raise ValueError(f'{name}: placement_extents {tuple(extents)} need x_min < x_max and y_min < y_max')
        if len(self._custom) >= _abi.MAX_CUSTOM_TASKS:
            raise ValueError(f'{name}: a batch holds at most {_abi.MAX_CUSTOM_TASKS} user-defined tasks')

    def _define(self, cls, base, obstacles, extents, claimed=True) -> int:
        """claimed=False: a definition restored by load_state_dict, under a stand-in class until task_id_of meets the
        user's class"""
        if _capturing():
            raise RuntimeError(f'defining the task {cls.__name__} synchronises: call task_id_of before the CUDA graph capture')
        self._check_definition(cls.__name__, base, obstacles, extents)
        d = _abi.SagTaskDef(base.task_id, (C.c_int32 * 4)(*obstacles), (C.c_double * 4)(*extents))
        tid = C.c_int32()
        self._lib.check(self._lib.L.sag_define_task(self._h, C.byref(d), C.byref(tid)))
        self._custom.append({'cls': cls, 'base': base, 'obstacles': list(obstacles), 'extents': list(extents),
                             'claimed': claimed})
        return tid.value

    def _definitions(self):
        return tuple((c['base'].task_id, tuple(c['obstacles']), tuple(c['extents'])) for c in self._custom)

    def _classes_by_id(self):
        by_id = {cls.task_id: cls for cls in _tasks.TASK_CLASSES}
        for k, c in enumerate(self._custom):
            by_id[_abi.NUM_TASKS + k] = c['cls']
        return by_id

    def _is_unsupervised(self, ids: torch.Tensor) -> torch.Tensor:
        """Which of `ids` run Unsupervised's logic (the registry task or a user-defined task based on it)."""
        unsup = [_tasks.Unsupervised.task_id] + [_abi.NUM_TASKS + k for k, c in enumerate(self._custom)
                                                 if c['base'] is _tasks.Unsupervised]
        return torch.isin(ids, torch.tensor(unsup, dtype=ids.dtype, device=ids.device))

    def render(self, mode='human'):
        raise NotImplementedError('rendering is outside the B200 hot path (reference: safe_adaptation_gym.py:109-111)')

    @property
    def observation(self) -> torch.Tensor:
        """safe_adaptation_gym.py:120-131: [obstacles lidar, objects lidar, goal lidar, sensors]"""
        L = self._lib
        L.check(L.L.sag_observe(self._h, self._p(self._obs), self._stream()))
        return self._out(self._obs)

    @property
    def lidar_observations(self) -> torch.Tensor:
        return self.observation[:, :3 * self.NUM_LIDAR_BINS]

    @property
    def action_space(self) -> Box:
        return self._action_space

    @property
    def observation_space(self) -> Box:
        if self._observation_space is None:  # safe_adaptation_gym.py:145-163
            lidar_size = 3 * self.NUM_LIDAR_BINS
            rest = self.obs_dim - lidar_size
            low = np.array([0.] * lidar_size + [-np.inf] * rest)
            high = np.array([1.] * lidar_size + [np.inf] * rest)
            self._observation_space = Box(low, high, shape=(self.obs_dim,), dtype=np.float32)
        return self._observation_space

    # ------------------------------------------------------------------------------------------
    # batched extras
    # ------------------------------------------------------------------------------------------
    def _as_action(self, action):
        on_device = (torch.is_tensor(action) and action.device.type == self.device.type
                     and (action.device.index or 0) == (self.device.index or 0))
        if not on_device and _capturing():
            raise RuntimeError('under CUDA graph capture the action must already be a tensor on the env\'s device '
                               f'({self.device}); a host or numpy action would record a copy from pageable memory')
        if not torch.is_tensor(action):
            action = torch.as_tensor(np.asarray(action, dtype=np.float32))
        act = action.to(device=self.device, dtype=torch.float32).reshape(self.num_envs, 2).contiguous()
        return act

    def _reset_all(self, new_task: bool, mask: Optional[torch.Tensor] = None, switch: bool = False):
        L = self._lib
        m = None
        if mask is not None:
            m = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        L.check(L.L.sag_reset(self._h, self._p(m), 0, 1 if new_task else 0, self._stream()))
        # world.py:75-78: drawn once per Task instance (also by the environments that took a queued task)
        if (new_task or switch or self._next_armed) and self.base_config['random_bound']:
            self._bound.copy_(self.get_field('task_f64')[14, :self.num_envs])  # in place: a CUDA graph may export it
        if self.device.type == 'cuda':
            torch.cuda.current_stream(self.device).synchronize()  # reset raises like the reference does (world.py:189)
        self._raise_recorded_errors('reset')

    def reset_envs(self, mask):
        """Reset only the environments where `mask` is true (vectorised-wrapper helper)."""
        self._forbid_capture('reset_envs')
        self._reset_all(new_task=False, mask=torch.as_tensor(mask))
        return self.observation

    def check_errors(self):
        """Raise the reference's exceptions for conditions recorded on the device since the last check.  This is how
        conditions recorded by CUDA graph replays of `step` surface: no Python runs during a replay."""
        self._forbid_capture('check_errors')
        if self.device.type == 'cuda':
            torch.cuda.current_stream(self.device).synchronize()
        self._raise_recorded_errors('step')
        flags = self.get_field('flags')[:self.num_envs]
        if bool(((flags & _abi.FLAG_RESAMPLE_FAILED) != 0).any()):
            raise ResamplingError('Failed to generate goal')  # go_to_goal.py:80

    _FIELDS = {'robot': (_abi.F_ROBOT, torch.float64, (6,)), 'objects': (_abi.F_OBJECTS, torch.float64, (6, _abi.MAX_SLOTS)),
               'task_f64': (_abi.F_TASK_F64, torch.float64, (15,)), 'task_i32': (_abi.F_TASK_I32, torch.int32, (10,)),
               'flags': (_abi.F_FLAGS, torch.uint8, ()), 'robot_ext': (_abi.F_ROBOT_EXT, torch.float64, (6,)),
               'gremlins': (_abi.F_GREMLINS, torch.float64, (2 + 3 * _abi.MAX_GREMLINS,)),
               'next_task': (_abi.F_NEXT_TASK, torch.int32, ())}

    def get_field(self, name: str) -> torch.Tensor:
        """Copy of an internal SoA state field, shape (*lead, stride) (see include/sag_b200.h SAG_F_*)."""
        fid, dt, lead = self._FIELDS[name]
        t = torch.empty(tuple(lead) + (self.stride,), dtype=dt, device=self.device)
        assert t.numel() * t.element_size() == self._lib.L.sag_field_bytes(self._h, fid)
        self._lib.check(self._lib.L.sag_read_field(self._h, fid, self._p(t), self._stream()))
        return t

    def set_field(self, name: str, value: torch.Tensor):
        self._forbid_capture('set_field')
        fid, dt, lead = self._FIELDS[name]
        t = torch.as_tensor(value).to(device=self.device, dtype=dt).contiguous()
        assert tuple(t.shape) == tuple(lead) + (self.stride,), (t.shape, lead, self.stride)
        self._lib.check(self._lib.L.sag_write_field(self._h, fid, self._p(t), self._stream()))
        if self.device.type == 'cuda':
            torch.cuda.current_stream(self.device).synchronize()  # `t` may be a temporary

    # ---- checkpoint / resume ------------------------------------------------------------------
    def state_dict(self) -> dict:
        """Everything a bit-exact continuation needs: the Philox key, every SoA state field (they carry the episode and
        in-step draw counters, the task ids, the queued next tasks and the cached clearance), and the host-side step
        budget.  The finished-episode statistics of `task_stats` are not part of it."""
        self._forbid_capture('state_dict')
        return {'seed': self._seed, 'num_envs': self.num_envs, 'robot': self.robot_name, 'custom_tasks': self._definitions(),
                'config': dict(self.base_config), 'env_id_base': self.env_id_base, 'max_episode_steps': self.max_episode_steps,
                'fields': {name: self.get_field(name).cpu() for name in self._FIELDS}}

    def load_state_dict(self, sd: dict):
        self._forbid_capture('load_state_dict')
        if sd['num_envs'] != self.num_envs or sd['robot'] != self.robot_name:
            raise ValueError('state_dict belongs to a different batch size / robot')
        for key, mine in (('config', dict(self.base_config)), ('env_id_base', self.env_id_base),
                          ('max_episode_steps', self.max_episode_steps)):
            if key in sd and sd[key] != mine:
                raise ValueError(f'state_dict was saved with a different {key}: {sd[key]!r} != {mine!r} (the continuation would not be bit-exact)')
        saved = tuple(sd.get('custom_tasks', ()))
        mine = self._definitions()
        if mine[:len(saved)] != saved[:len(mine)]:
            raise ValueError(f'state_dict defines the user-defined tasks {saved!r}, which conflict with this batch\'s '
                             f'{mine!r}')
        for base_id, obstacles, extents in saved[len(mine):]:
            base = {c.task_id: c for c in _tasks.TASK_CLASSES}[base_id]
            cls = type(f'{base.__name__}Custom{len(self._custom)}', (base,), {
                'obstacles': property(lambda self, o=list(obstacles): list(o)),
                'placement_extents': property(lambda self, x=tuple(extents): x)})
            self._define(cls, base, list(obstacles), list(extents), claimed=False)
        self.seed(sd['seed'])
        for name, value in sd['fields'].items():
            self.set_field(name, value)
        if 'next_task' not in sd['fields']:   # saved before tasks could be queued: nothing queued
            self.set_field('next_task', torch.full((self.stride,), -1, dtype=torch.int32))
        if bool((sd['fields'].get('next_task', torch.full((1,), -1)) != -1).any()):
            self._next_armed = True
        ids = sd['fields']['task_i32'][0, :self.num_envs].to(torch.int32)
        self._tasks_from_ids(ids)
        self._any_unsupervised = bool(self._is_unsupervised(ids).any())
        self._observation_space = None
        if self.base_config['random_bound']:
            self._bound.copy_(self.get_field('task_f64')[14, :self.num_envs])  # in place: a CUDA graph may export it

    def rollout(self, k_steps: int):
        """K steps per launch with on-device Philox U(-1,1) actions; returns the last step's outputs."""
        L = self._lib
        L.check(L.L.sag_rollout(self._h, int(k_steps), self._p(self._obs), self._p(self._reward), self._p(self._cost),
                                self._p(self._done), self._stream()))
        return (self._out(self._obs), self._out(self._reward), self._done.to(torch.bool),
                {'cost': self._cost.to(torch.float32), 'bound': self._out(self._bound)})

    def task_stats(self, reset: bool = False) -> torch.Tensor:
        """[14 + user-defined tasks, 3] float64: per-task id (sum of finished-episode returns, sum of costs, #episodes)
        on this device.  Row 14 + k is the k-th user-defined task of this batch (``task_id_of``): ranks that reduce
        these rows together (``stats.reduce_task_stats``) must define the same tasks in the same order."""
        # as many rows as the library writes (a task may also have been defined through the C ABI on this handle)
        L = self._lib.L
        rows = L.sag_num_task_ids(self._h) if hasattr(L, 'sag_num_task_ids') else _abi.NUM_TASKS
        out = torch.zeros((rows, 3), dtype=torch.float64, device=self.device)
        self._lib.check(self._lib.L.sag_task_stats(self._h, self._p(out), 1 if reset else 0, self._stream()))
        return out
