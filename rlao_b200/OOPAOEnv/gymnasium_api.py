"""Gymnasium-style face of the Shack-Hartmann environment.

The reference documents this signature on its Pyramid environments (MAIN_CODE/OOPAOEnv/OOPAOEnv_VPG.py:117-137
`reset(seed, options) -> (obs, info)`, :553-611 `step(action) -> (obs, reward, terminated, truncated, info)`):
the observation is a stack of the last `n_history` reconstructed-command images (newest first, `roll_buffer`
:660-682), actions pass through a FIFO of `delay` frames (:560-566), the reward is the Strehl ratio (:597-601) and
the episode never terminates by itself.  This adapter gives the same face to `OOPAOEnvRazor.OOPAO` (SURVEY.md
section 8 b) without adding work to the step: history and delay are ring buffers on the device.

`gymnasium` itself is not a dependency; `observation_space` / `action_space` are plain `Box` records with the
fields RL libraries read (`low`, `high`, `shape`, `dtype`).
"""
import collections

import numpy as np
import torch

Box = collections.namedtuple("Box", ["low", "high", "shape", "dtype"])


class GymnasiumSH:
    """env = GymnasiumSH(oopao_env, n_history=20, delay=1, episode_length=None)

    obs: float32 [n_envs, n_history, nAct, nAct] on the device ([n_history, nAct, nAct] for one environment);
    action: [n_envs, nAct, nAct] image or [n_envs, nValidAct] vector, micro-metres (scaled by 1e-6 in the step
    kernel like OOPAOEnv_VPG.py:566).  `truncated` turns True after `episode_length` steps when one is given
    (the reference leaves truncation to a TimeLimit wrapper).
    """

    metadata = {"render_modes": []}

    def __init__(self, env, n_history=20, delay=1, episode_length=None):
        self.env = env
        self.n_history = int(n_history)
        self.d = int(delay)
        self.episode_length = episode_length
        nA, B = env.nActuator, env.n_envs
        lead = () if B == 1 else (B,)
        self.observation_space = Box(-np.inf, np.inf, lead + (self.n_history, nA, nA), np.float32)
        self.action_space = Box(-1.0, 1.0, lead + (nA, nA), np.float32)
        self._hist = torch.zeros((B, self.n_history, nA, nA), dtype=torch.float32, device=env.device)
        self._fifo = torch.zeros((max(self.d, 1), B, nA, nA), dtype=torch.float32, device=env.device)
        self._t = 0
        self._rng = np.random.RandomState()

    def __getattr__(self, name):
        return getattr(self.__dict__["env"], name)

    # ---- helpers ------------------------------------------------------------------------------------------
    def _push(self, obs):
        """roll_buffer (OOPAOEnv_VPG.py:660-682): newest image at index 0."""
        self._hist = torch.roll(self._hist, shifts=1, dims=1)
        self._hist[:, 0] = obs.reshape(self.env.n_envs, *obs.shape[-2:])

    def _out(self):
        h = self._hist[0] if self.env.n_envs == 1 else self._hist
        return h.clone()

    # ---- gymnasium API --------------------------------------------------------------------------------------
    def reset(self, seed=None, options=None):
        """OOPAOEnv_VPG.py:117-137: flat DM, new phase screens, WFS measurement of the bare atmosphere."""
        if seed is not None:
            self._rng = np.random.RandomState(seed)
        e = self.env
        e.dm.coefs = 0
        e.dm_prev = 0
        e.atm.generateNewPhaseScreen(seed=int(self._rng.randint(0, 100000)))
        e.tel * e.wfs
        e.SR = []
        self._fifo.zero_()
        self._hist.zero_()
        self._t = 0
        self._push(e.reset_soft())
        return self._out(), {}

    def step(self, action):
        """OOPAOEnv_VPG.py:553-611."""
        e = self.env
        a = torch.as_tensor(action, dtype=torch.float32, device=e.device)
        if a.shape[-1] == e.dm.nValidAct and a.shape[-2:] != (e.nActuator, e.nActuator):
            a = e.vec_to_img(a)                                          # :558-559
        a = a.reshape(e.n_envs, e.nActuator, e.nActuator)
        if self.d > 0:                                                   # :561-566 FIFO of `delay` frames
            slot = self._t % self.d
            delayed = self._fifo[slot].clone()
            self._fifo[slot] = a
        else:
            delayed = a
        obs, _, strehl, _, info = e._step_views(self._t, delayed)
        self._t += 1
        self._push(obs)
        reward = strehl.clone() if torch.is_tensor(strehl) else strehl   # :597-601 reward = Strehl
        truncated = self.episode_length is not None and self._t >= self.episode_length
        return self._out(), reward, False, bool(truncated), {"strehl": reward}

    def close(self):
        pass


class GymnasiumVectorSH:
    """env = GymnasiumVectorSH(oopao_env, n_history=20, delay=1, episode_length=None, stagger_episodes=False)

    The vector-env face of the same environment (Gymnasium's vector API, SB3 VecEnv, CleanRL, TorchRL): every one of the
    n_envs environments runs its own episode.  step(actions) returns obs [B, n_history, nAct, nAct] and reward [B] on the
    device, terminated [B] (always False) and truncated [B] as host bool arrays, and info; `truncated` comes from
    per-environment step counters kept on the host and `episode_length`.

    Next-step autoreset: an environment truncated at call t is reset at call t+1 through OOPAO.reset_envs (new screens,
    flat mirror; the other environments continue bit for bit).  At that call its action is ignored (zero rows), its
    history stack and delay FIFO rows are cleared, and it returns the first observation of its new episode with reward 0
    and truncated False.  reset(options={"reset_mask": mask}) resets the masked environments the same way (their
    observation rows are zero until their next step measures the new episode); reset() without a mask is the full reset
    of GymnasiumSH.  stagger_episodes=True starts environment e at step e * episode_length // B, so that resets spread
    evenly over the episode.  Each reset call takes one seed from the wrapper's RNG: a seeded run is reproducible."""

    metadata = {"render_modes": [], "autoreset_mode": "NextStep"}

    def __init__(self, env, n_history=20, delay=1, episode_length=None, stagger_episodes=False):
        self.env = env
        self.n_history = int(n_history)
        self.d = int(delay)
        self.episode_length = None if episode_length is None else int(episode_length)
        self.stagger_episodes = bool(stagger_episodes)
        nA, B = env.nActuator, env.n_envs
        self.num_envs = B
        self.single_observation_space = Box(-np.inf, np.inf, (self.n_history, nA, nA), np.float32)
        self.single_action_space = Box(-1.0, 1.0, (nA, nA), np.float32)
        self.observation_space = Box(-np.inf, np.inf, (B, self.n_history, nA, nA), np.float32)
        self.action_space = Box(-1.0, 1.0, (B, nA, nA), np.float32)
        self._hist = torch.zeros((B, self.n_history, nA, nA), dtype=torch.float32, device=env.device)
        self._fifo = torch.zeros((max(self.d, 1), B, nA, nA), dtype=torch.float32, device=env.device)
        self._t = 0
        self._steps = np.zeros(B, dtype=np.int64)          # steps taken in the current episode, per environment
        self._pending = np.zeros(B, dtype=bool)            # truncated at the last call: reset at the next one
        self._rng = np.random.RandomState()

    def __getattr__(self, name):
        return getattr(self.__dict__["env"], name)

    def _start_steps(self):
        B, L = self.num_envs, self.episode_length
        if self.stagger_episodes and L is not None:
            return np.arange(B, dtype=np.int64) * L // B
        return np.zeros(B, dtype=np.int64)

    def _reset_subset(self, ids):
        """OOPAO.reset_envs of host indices `ids`, the wrapper's rows cleared; returns the device index tensor."""
        idx = self.env.reset_envs(ids, int(self._rng.randint(0, 2 ** 31 - 1))).long()
        self._hist.index_fill_(0, idx, 0.0)
        self._fifo.index_fill_(1, idx, 0.0)
        self._steps[ids] = 0
        self._pending[ids] = False
        return idx

    def reset(self, seed=None, options=None):
        """Full reset (GymnasiumSH.reset) without a mask; options={"reset_mask": mask [B] (host or device bool)}: only those."""
        if seed is not None:
            self._rng = np.random.RandomState(seed)
        mask = (options or {}).get("reset_mask")
        if mask is None:
            e = self.env
            e.dm.coefs = 0
            e.dm_prev = 0
            e.atm.generateNewPhaseScreen(seed=int(self._rng.randint(0, 100000)))
            e.tel * e.wfs
            e.SR = []
            self._fifo.zero_()
            self._hist.zero_()
            self._t = 0
            self._steps = self._start_steps()
            self._pending[:] = False
            obs = e.reset_soft()
            self._hist[:, 0] = obs.reshape(e.n_envs, *obs.shape[-2:])
            return self._hist.clone(), {}
        mask = mask.cpu().numpy() if torch.is_tensor(mask) else np.asarray(mask)
        if mask.shape != (self.num_envs,) or mask.dtype != bool:
            raise ValueError(f"reset_mask must be a bool array of shape ({self.num_envs},)")
        ids = np.nonzero(mask)[0]
        if ids.size:
            self._reset_subset(ids)
        return self._hist.clone(), {}

    def step(self, actions):
        """GymnasiumSH.step for every environment, with next-step autoreset."""
        e = self.env
        a = torch.as_tensor(actions, dtype=torch.float32, device=e.device)
        if a.shape[-1] == e.dm.nValidAct and a.shape[-2:] != (e.nActuator, e.nActuator):
            a = e.vec_to_img(a)
        a = a.reshape(e.n_envs, e.nActuator, e.nActuator)
        resetting = self._pending.copy()
        idx = None
        if resetting.any():
            idx = self._reset_subset(np.nonzero(resetting)[0])
            a = a.index_fill(0, idx, 0.0)                                 # the action of a resetting environment is ignored
        if self.d > 0:
            slot = self._t % self.d
            delayed = self._fifo[slot].clone()
            self._fifo[slot] = a
        else:
            delayed = a
        obs, _, strehl, _, info = e._step_views(self._t, delayed)
        self._t += 1
        self._hist = torch.roll(self._hist, shifts=1, dims=1)
        self._hist[:, 0] = obs.reshape(e.n_envs, *obs.shape[-2:])
        strehl = strehl.reshape(e.n_envs).clone()
        reward = strehl.clone()
        if idx is not None:
            reward.index_fill_(0, idx, 0.0)
        self._steps += ~resetting
        truncated = (self._steps >= self.episode_length) if self.episode_length is not None else np.zeros(self.num_envs, dtype=bool)
        self._pending = truncated.copy()
        terminated = np.zeros(self.num_envs, dtype=bool)
        return self._hist.clone(), reward, terminated, truncated, {"strehl": strehl, "autoreset": resetting}

    def close(self):
        pass
