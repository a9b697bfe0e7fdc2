"""RL-library adapters for the batched environments (reference: ``fluidgym/integration/{gymnasium,pettingzoo}.py``,
``integration/sb3/vec_env.py``).

The reference converts the observation of ONE environment to numpy per call and maps the agents of one multi-agent
environment onto the slots of a Stable-Baselines3 ``VecEnv``.  A batched environment already is a vector of
environments, so here

* ``VecFluidEnv`` exposes ``n_envs x n_agents`` slots (environment-major) with the ``VecEnv`` call protocol
  (``reset / step_async / step_wait / get_attr / set_attr / env_is_wrapped / close``, auto-reset with
  ``terminated_observation`` as in vec_env.py:96-152), one device->host copy per observation key and step;
* ``GymFluidEnv`` / ``PettingZooFluidEnv`` are the single-environment views (``n_envs == 1``) with the reference's
  constructor checks and error messages (gymnasium.py:22-37, pettingzoo.py:27-49).

None of the three libraries is imported: the classes are duck-typed (SB3 only needs the attributes and methods below;
``stable_baselines3.common.vec_env.VecEnv`` is mixed in as a base class when it is importable so that ``isinstance``
checks inside SB3 pass).  The solver path is untouched by this module.
"""
from __future__ import annotations

from typing import Any

import numpy as np
import torch

try:                                                     # pragma: no cover - not installed in the build image
    from stable_baselines3.common.vec_env import VecEnv as _SB3VecEnv
except Exception:                                        # noqa: BLE001
    _SB3VecEnv = object


def _np(t):
    return t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def _np_tree(x):
    return {k: _np(v) for k, v in x.items()} if isinstance(x, dict) else _np(x)


def _device(env):
    return getattr(env, "device", None) or getattr(env, "cuda_device")


def _check_render_mode(render_mode):
    if render_mode is not None and render_mode != "rgb_array":
        raise ValueError(f"Unsupported render mode: {render_mode}. Only 'rgb_array' is supported.")


class VecFluidEnv(_SB3VecEnv):
    """SB3 ``VecEnv`` protocol over a batched environment: slot ``e * n_agents + a`` = agent ``a`` of environment ``e``."""

    metadata = {"render_modes": ["rbg_array"]}

    def __init__(self, env, auto_reset: bool = True, render_mode: str | None = None):
        _check_render_mode(render_mode)
        self._env = env
        self._auto_reset = auto_reset
        self.n_envs_batch = int(getattr(env, "n_envs", 1))
        self.n_agents = int(env.n_agents) if getattr(env, "use_marl", False) else 1
        self.num_envs = self.n_envs_batch * self.n_agents
        self.observation_space = env.observation_space
        self.action_space = env.action_space
        self._actions = None
        self.render_mode = render_mode

    # --- layout helpers -----------------------------------------------------------------------------
    def _flat(self, x):
        """[B, (n_agents,) ...] -> [num_envs, ...]"""
        a = _np(x)
        if self.n_agents > 1:
            return a.reshape((self.num_envs,) + a.shape[2:])
        return a

    def _flat_obs(self, obs):
        return {k: self._flat(v) for k, v in obs.items()} if isinstance(obs, dict) else self._flat(obs)

    # --- VecEnv protocol ----------------------------------------------------------------------------
    def reset(self, seed: int | None = None, randomize: bool | None = None):
        obs, _ = self._env.reset(seed=seed, randomize=randomize)
        return self._flat_obs(obs)

    def step_async(self, actions) -> None:
        a = torch.as_tensor(np.asarray(actions), dtype=torch.float32, device=_device(self._env))
        shape = tuple(self.action_space.shape)
        if self.n_agents > 1:
            a = a.reshape((self.n_envs_batch, self.n_agents) + shape)
        else:
            a = a.reshape((self.n_envs_batch,) + shape)
        self._actions = a

    def step_wait(self):
        obs, reward, term, trunc, info = self._env.step(self._actions)
        obs_np = self._flat_obs(obs)
        r = _np(reward)
        if self.n_agents > 1 and r.ndim == 1:           # global reward only: every agent of an environment receives it
            r = np.repeat(r, self.n_agents)
        rewards = r.reshape(self.num_envs).astype(np.float32)
        done = bool(term) or bool(trunc)
        dones = np.full(self.num_envs, done, dtype=bool)
        info_np = _np_tree(info)
        infos: list[dict[str, Any]] = []
        for i in range(self.num_envs):
            e = i // self.n_agents
            d = {}
            for k, v in info_np.items():
                d[k] = v[e] if isinstance(v, np.ndarray) and v.ndim >= 1 and v.shape[0] == self.n_envs_batch else v
            d["TimeLimit.truncated"] = bool(trunc) and not bool(term)
            infos.append(d)
        if done and self._auto_reset:                   # vec_env.py:140-150
            for i in range(self.num_envs):
                infos[i]["terminated_observation"] = ({k: v[i] for k, v in obs_np.items()} if isinstance(obs_np, dict) else obs_np[i])
            obs_np = self.reset()
        return obs_np, rewards, dones, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def get_attr(self, attr_name: str, indices=None) -> list[Any]:
        return [getattr(self._env, attr_name)] * self.num_envs

    def set_attr(self, attr_name: str, value: Any, indices=None) -> None:
        setattr(self._env, attr_name, value)

    def env_is_wrapped(self, wrapper_class, indices=None) -> list[bool]:
        return [False] * self.num_envs

    def env_method(self, method_name: str, *method_args, indices=None, **method_kwargs):
        raise NotImplementedError

    def get_images(self) -> list:
        """One uint8 [H, W, 3] image per slot (the agents of an environment share its image); ``None`` per slot unless
        ``render_mode == "rgb_array"``.  One batched ``env.render()`` and one device->host copy."""
        if self.render_mode != "rgb_array":
            return [None] * self.num_envs
        imgs = _np(self._env.render())
        return [imgs[i // self.n_agents] for i in range(self.num_envs)]

    def seed(self, seed: int | None = None):
        if seed is not None:
            self._env.seed(seed)
        return [seed] * self.num_envs

    def close(self) -> None:
        pass

    @property
    def unwrapped(self):
        return getattr(self._env, "unwrapped", self._env)

    def train(self) -> None:
        self._env.train()

    def val(self) -> None:
        self._env.val()

    def test(self) -> None:
        self._env.test()


def _single(env, who: str):
    if int(getattr(env, "n_envs", 1)) != 1:
        raise ValueError(f"{who} wraps one environment: construct it with n_envs=1 (use VecFluidEnv for batches).")


class GymFluidEnv:
    """``gymnasium.Env`` call protocol for one single-agent environment (gymnasium.py:14-214): numpy in, numpy out."""

    metadata = {"render_modes": ["rbg_array"], "render_fps": 24}

    def __init__(self, env, render_mode: str | None = None):
        if getattr(env, "use_marl", False):
            raise ValueError("GymFluidEnv does not support multi-agent environments. Please use a single-agent environment.")
        _check_render_mode(render_mode)
        _single(env, "GymFluidEnv")
        self.render_mode = render_mode
        self._env = env
        self.action_space = env.action_space
        self.observation_space = env.observation_space

    @staticmethod
    def _squeeze(x):
        return {k: _np(v)[0] for k, v in x.items()} if isinstance(x, dict) else _np(x)[0]

    def step(self, action):
        a = torch.as_tensor(np.asarray(action), dtype=torch.float32, device=_device(self._env)).unsqueeze(0)
        obs, reward, terminated, truncated, info = self._env.step(a)
        info_np = {k: np.array(_np(v)).reshape(-1)[0] if np.size(_np(v)) == 1 else _np(v)[0] for k, v in info.items()}
        return self._squeeze(obs), float(_np(reward).reshape(-1)[0]), bool(terminated), bool(truncated), info_np

    def reset(self, *, seed: int | None = None, options: dict | None = None, randomize: bool | None = None):
        obs, info = self._env.reset(seed=seed, randomize=randomize)
        return self._squeeze(obs), {k: _np(v) for k, v in info.items()}

    def render(self):
        """uint8 [H, W, 3] numpy image of the environment with ``render_mode == "rgb_array"``, otherwise ``None``."""
        if self.render_mode != "rgb_array":
            return None
        return _np(self._env.render()[0])

    def close(self):
        pass

    @property
    def unwrapped(self):
        return getattr(self._env, "unwrapped", self._env)


class PettingZooFluidEnv:
    """``pettingzoo.ParallelEnv`` call protocol for one multi-agent environment (pettingzoo.py:14-203): dictionaries keyed
    by ``agent_<i>``."""

    metadata = {"render_modes": ["rbg_array"], "name": "fluidgym_b200"}

    def __init__(self, env):
        if not getattr(env, "use_marl", False) or env.n_agents <= 1:
            raise ValueError("PettingZooFluidEnv can only be used with MARL fluid environments with multiple agents.")
        _single(env, "PettingZooFluidEnv")
        self._env = env
        self.possible_agents = [f"agent_{i}" for i in range(env.n_agents)]
        self.agents = list(self.possible_agents)

    def observation_space(self, agent):
        return self._env.observation_space

    def action_space(self, agent):
        return self._env.action_space

    def _per_agent(self, obs):
        if isinstance(obs, dict):
            arr = {k: _np(v)[0] for k, v in obs.items()}
            return {a: {k: v[i] for k, v in arr.items()} for i, a in enumerate(self.agents)}
        arr = _np(obs)[0]
        return {a: arr[i] for i, a in enumerate(self.agents)}

    def reset(self, seed: int | None = None, options: dict | None = None, randomize: bool | None = None):
        self.agents = list(self.possible_agents)
        obs, _ = self._env.reset(seed=seed, randomize=randomize)
        return self._per_agent(obs), {a: {} for a in self.agents}

    def step(self, actions: dict):
        a = np.stack([np.asarray(actions[ag], dtype=np.float32) for ag in self.agents])
        t = torch.as_tensor(a, device=_device(self._env)).reshape((1, len(self.agents)) + tuple(self._env.action_space.shape))
        obs, reward, terminated, truncated, info = self._env.step(t)
        r = _np(reward)[0]
        rewards = {ag: float(r[i]) for i, ag in enumerate(self.agents)}
        info_np = {k: _np(v)[0] for k, v in info.items()}
        infos = {ag: info_np for ag in self.agents}
        terms = {ag: bool(terminated) for ag in self.agents}
        truncs = {ag: bool(truncated) for ag in self.agents}
        observations = self._per_agent(obs)
        if terminated or truncated:
            self.agents = []
        return observations, rewards, terms, truncs, infos

    def seed(self, seed: int) -> None:
        self._env.seed(seed)

    def close(self):
        pass

    @property
    def unwrapped(self):
        return getattr(self._env, "unwrapped", self._env)


# ------------------------------------------------------------------------------------------------
# TorchRL (reference: fluidgym/integration/torchrl.py:87-278)
# ------------------------------------------------------------------------------------------------
try:                                                     # pragma: no cover - not installed in the build image
    from tensordict import TensorDict as _TensorDict
    from torchrl.data.tensor_specs import Bounded as _Bounded, Categorical as _Categorical, Composite as _Composite, \
        Unbounded as _Unbounded
    from torchrl.envs import EnvBase as _TorchRLEnvBase
    _HAVE_TORCHRL = True
except Exception:                                        # noqa: BLE001
    _HAVE_TORCHRL = False

    class _TorchRLEnvBase:                               # the part of EnvBase's constructor contract this adapter uses
        def __init__(self, device=None, batch_size=()):
            self.device, self.batch_size = device, torch.Size(batch_size)


class SpecLike:
    """Stand-in for a TorchRL tensor spec when torchrl is not installed: shape / dtype / bounds, nothing else."""

    def __init__(self, shape, dtype=torch.float32, low=None, high=None, device=None):
        self.shape, self.dtype, self.low, self.high, self.device = torch.Size(shape), dtype, low, high, device

    def __repr__(self):
        return f"SpecLike(shape={tuple(self.shape)}, dtype={self.dtype})"


class TorchRLFluidEnv(_TorchRLEnvBase):
    """TorchRL ``EnvBase`` over a batched environment.

    The reference exposes ONE environment: batch size ``()`` single-agent, ``(n_agents,)`` multi-agent (the agents as a virtual
    batch, torchrl.py:87-100).  A batched environment is a real batch: batch size ``(n_envs,)`` or ``(n_envs, n_agents)``, all
    tensors stay on the environment's device (no numpy round trip).  Same ``_step / _reset / _set_seed`` protocol and the same
    spec layout (observation keys as a Composite, reward / done / terminated / truncated with a trailing unit dimension).
    ``from_pixels`` adds ``"pixels"``, the environment's ``render()`` as uint8 ``(*batch_size, H, W, 3)``, to
    the observation spec and to every reset / step; the agents of one environment share its image (an expanded view)."""

    def __init__(self, env, from_pixels: bool = False):
        if from_pixels and not callable(getattr(env, "render", None)):
            raise NotImplementedError(f"from_pixels: {type(env).__name__} has no render()")
        self._from_pixels = bool(from_pixels)
        n_envs = int(getattr(env, "n_envs", 1))
        self._n_agents = int(env.n_agents) if getattr(env, "use_marl", False) else None
        batch = (n_envs,) if self._n_agents is None else (n_envs, self._n_agents)
        super().__init__(device=_device(env), batch_size=torch.Size(batch))
        self._env = env
        self._make_spec()

    def _box(self, space, lead):
        low = torch.as_tensor(np.broadcast_to(space.low, space.shape).copy(), dtype=torch.float32, device=self.device)
        high = torch.as_tensor(np.broadcast_to(space.high, space.shape).copy(), dtype=torch.float32, device=self.device)
        shape = torch.Size((*lead, *space.shape))
        unbounded = bool(np.all(np.isinf(space.low)) and np.all(np.isinf(space.high)))
        if not _HAVE_TORCHRL:
            return SpecLike(shape, low=None if unbounded else low.expand(shape), high=None if unbounded else high.expand(shape), device=self.device)
        if unbounded:
            return _Unbounded(shape=shape, dtype=torch.float32, device=self.device)
        return _Bounded(low=low.expand(shape).clone(), high=high.expand(shape).clone(), shape=shape, dtype=torch.float32, device=self.device)

    def _make_spec(self) -> None:                         # torchrl.py:128-190
        lead = tuple(self.batch_size)
        obs_space = self._env.observation_space
        sub = obs_space.spaces if hasattr(obs_space, "spaces") else {"observation": obs_space}
        obs = {k: self._box(v, lead) for k, v in sub.items()}
        if self._from_pixels:
            H, W = self._pixels().shape[-3:-1]
            shape = torch.Size((*lead, H, W, 3))
            obs["pixels"] = _Bounded(low=0, high=255, shape=shape, dtype=torch.uint8, device=self.device) if _HAVE_TORCHRL else \
                SpecLike(shape, dtype=torch.uint8, low=0, high=255, device=self.device)
        flag = (lambda: SpecLike((*lead, 1), dtype=torch.bool, device=self.device)) if not _HAVE_TORCHRL else \
            (lambda: _Categorical(n=2, shape=torch.Size((*lead, 1)), dtype=torch.bool, device=self.device))
        if _HAVE_TORCHRL:                                # pragma: no cover
            self.observation_spec = _Composite(obs, shape=self.batch_size)
            self.state_spec = self.observation_spec.clone()
            self.reward_spec = _Unbounded(shape=torch.Size((*lead, 1)), dtype=torch.float32, device=self.device)
            self.done_spec = _Composite(done=flag(), terminated=flag(), truncated=flag(), shape=self.batch_size)
        else:
            self.observation_spec = obs
            self.state_spec = dict(obs)
            self.reward_spec = SpecLike((*lead, 1), device=self.device)
            self.done_spec = {"done": flag(), "terminated": flag(), "truncated": flag()}
        self.action_spec = self._box(self._env.action_space, lead)

    def _pixels(self) -> torch.Tensor:
        img = self._env.render()                                        # [n_envs, H, W, 3]
        if self._n_agents is not None:
            img = img[:, None].expand(img.shape[0], self._n_agents, *img.shape[1:])
        return img

    def _observe(self, obs) -> dict:
        if not isinstance(obs, dict):
            obs = {"observation": obs}
        return {**obs, "pixels": self._pixels()} if self._from_pixels else obs

    def _td(self, data: dict):
        return _TensorDict(data, batch_size=self.batch_size) if _HAVE_TORCHRL else dict(data)

    def _flag(self, flag: bool) -> torch.Tensor:
        return torch.full((*self.batch_size, 1), bool(flag), dtype=torch.bool, device=self.device)

    def _step(self, tensordict):                          # torchrl.py:205-244
        with torch.no_grad():
            obs, reward, term, trunc, _ = self._env.step(tensordict["action"])
            obs = self._observe(obs)
        reward = reward.reshape(*self.batch_size, 1)
        return self._td({**obs, "reward": reward, "done": self._flag(term or trunc), "terminated": self._flag(term),
                         "truncated": self._flag(trunc)})

    def _reset(self, tensordict=None, **kwargs):          # torchrl.py:246-268
        obs, _ = self._env.reset()
        return self._td(self._observe(obs))

    def _set_seed(self, seed: int) -> None:               # torchrl.py:270-278
        self._env.seed(seed)

    if not _HAVE_TORCHRL:                                 # EnvBase provides these when torchrl is installed
        def reset(self, tensordict=None, **kwargs):
            return self._reset(tensordict, **kwargs)

        def step(self, tensordict):
            out = self._step(tensordict)
            return {**tensordict, "next": out}

        def set_seed(self, seed: int):
            self._set_seed(seed)
            return seed
