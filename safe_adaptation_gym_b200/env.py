"""Batched drop-in variant of ``SafeAdaptationGym`` (reference: safe_adaptation_gym/safe_adaptation_gym.py:21-257).

Same method names and argument meaning as the reference env, with a leading batch dimension:

    obs[N, D], reward[N], done[N], info{'cost'[N], 'bound'[N]} = env.step(actions[N, nu])
    obs[N, D] = env.reset(options={'task': task_or_list_of_tasks})

Returned tensors are fresh copies by default, like the arrays the reference returns; ``copy_outputs=False`` hands out the
internal output buffers instead (valid until the next call -- the zero-copy mode for throughput loops).
With ``max_episode_steps > 0`` the env auto-resets like a vectorised gym wrapper: an environment whose episode ended
(time limit, or done after a physics error) is reset inside ``step``; its row of ``obs`` is the FIRST observation of the
new episode, ``done`` is True for it and ``info['truncated']`` marks the time-limit endings.

``step`` (both output modes, with or without auto-reset), ``rollout`` and ``observation`` may be recorded in a CUDA graph
(``torch.cuda.graph``), together with the policy that computes the actions; every replay behaves like issuing the same
calls again.  ``seed``, ``set_task`` and ``load_state_dict`` between replays are seen by the graph, except that a
``set_task`` which changes whether any environment runs ``Unsupervised`` changes the reward buffer ``step`` records:
capture again after it.  No Python runs during a replay, so errors recorded by replayed steps are raised by
``check_errors()``.  The methods that synchronise raise ``RuntimeError`` while a capture is open.

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
        self._bound = torch.full((n,), float(cfg['max_bound']), dtype=torch.float64, device=dev)
        self._task_ids = None
        self._tasks = None
        self._any_unsupervised = False
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

    def set_task(self, task):
        """safe_adaptation_gym.py:165-168.  `task`: a Task, or a sequence of N Tasks (one per environment).

        A CUDA graph that records ``step`` must be captured again when this changes whether any environment runs
        ``Unsupervised`` (its reward is a pair, written to another buffer)."""
        self._forbid_capture('set_task')
        if isinstance(task, _tasks.Task):
            task_list = [task] * self.num_envs
        else:
            task_list = list(task)
            if len(task_list) != self.num_envs:
                raise ValueError(f'need {self.num_envs} tasks, got {len(task_list)}')
        for t in task_list:
            if t.name in _tasks.DEVICE_UNSUPPORTED:
                raise NotImplementedError(f"task '{t.name}' is not implemented on the device path yet")
        ids = torch.tensor([t.task_id for t in task_list], dtype=torch.int32)
        self._tasks = task_list
        self._task_ids = ids.to(self.device)
        self._any_unsupervised = bool((ids == _tasks.Unsupervised.task_id).any())
        self._lib.check(self._lib.L.sag_set_tasks(self._h, self._p(self._task_ids), self._stream()))
        self._observation_space = None
        self._reset_all(new_task=True)

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

    def _reset_all(self, new_task: bool, mask: Optional[torch.Tensor] = None):
        L = self._lib
        m = None
        if mask is not None:
            m = mask.to(device=self.device, dtype=torch.uint8).contiguous()
        L.check(L.L.sag_reset(self._h, self._p(m), 0, 1 if new_task else 0, self._stream()))
        if new_task and self.base_config['random_bound']:  # world.py:75-78: drawn once per Task instance
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
               'gremlins': (_abi.F_GREMLINS, torch.float64, (2 + 3 * _abi.MAX_GREMLINS,))}

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
        in-step draw counters, the task ids and the cached clearance), and the host-side step budget.  The
        finished-episode statistics of `task_stats` are not part of it."""
        self._forbid_capture('state_dict')
        return {'seed': self._seed, 'num_envs': self.num_envs, 'robot': self.robot_name,
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
        self.seed(sd['seed'])
        for name, value in sd['fields'].items():
            self.set_field(name, value)
        ids = sd['fields']['task_i32'][0, :self.num_envs].to(torch.int32)
        by_id = {cls.task_id: cls for cls in _tasks.TASK_CLASSES}
        self._tasks = [by_id[int(i)]() for i in ids.tolist()]
        self._task_ids = ids.to(self.device)
        self._any_unsupervised = bool((ids == _tasks.Unsupervised.task_id).any())
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
        """[14, 3] float64: per-task (sum of finished-episode returns, sum of costs, #episodes) on this device."""
        out = torch.zeros((_abi.NUM_TASKS, 3), dtype=torch.float64, device=self.device)
        self._lib.check(self._lib.L.sag_task_stats(self._h, self._p(out), 1 if reset else 0, self._stream()))
        return out
