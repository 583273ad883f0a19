"""Mirror of MAIN_CODE/PO4AO/util_simple.py for the environment boundary: TorchWrapper, TimeDelayEnv and the
GPU-resident EfficientExperienceReplay (sample_contiguous semantics of :103-111)."""
import torch


class _Wrapper:
    """Attribute-forwarding wrapper (the role gym.Wrapper plays in the reference)."""

    def __init__(self, env):
        self.env = env
        self._env = env

    def __getattr__(self, name):
        return getattr(self.__dict__["env"], name)


class TimeDelayEnv(_Wrapper):
    """util_simple.py:25-52: FIFO of `delay` zero actions in front of env.step."""

    def __init__(self, env, delay):
        super().__init__(env)
        self.d = delay
        self._zero()

    def _zero(self):
        e = self._env
        shape = (e.nActuator, e.nActuator) if e.n_envs == 1 else (e.n_envs, e.nActuator, e.nActuator)
        self.action_buffer = [torch.zeros(shape, dtype=torch.float32, device=e.device) for _ in range(self.d)]

    def reset_soft(self):
        obs = self._env.reset_soft()
        self._zero()
        return obs

    def step(self, i, action):
        self.action_buffer.append(torch.as_tensor(action, dtype=torch.float32, device=self._env.device))
        out = self._env.step(i, self.action_buffer[0])
        del self.action_buffer[0]
        return out


class TorchWrapper(_Wrapper):
    """util_simple.py:201-221.  The reference converts torch -> numpy -> torch around a host simulation and hands
    back CPU float32 tensors; this wrapper keeps that contract with pinned staging buffers and asynchronous copies
    (`host_io=True`, default), or keeps everything on the device (`host_io=False`) for on-GPU policies."""

    def __init__(self, env, host_io=True, lookahead=False):
        """lookahead (host_io only, opt-in): the observation of frame t+1 does not depend on the action of step t+1 (one
        frame of DM lag), so `step(t, a_t)` applies a_t and then already runs frame t+1 (WFS, reconstruction), starts
        its download and issues the atmosphere of frame t+2; the next call returns obs(t+1) without waiting for the
        GPU.  Same numbers as the strict path, but the simulation runs ahead of what was returned: call `flush()` (or
        `reset_soft()`) before touching the environment's objects between steps."""
        super().__init__(env)
        self.host_io = host_io
        self.lookahead = bool(lookahead)
        self._ahead = None
        self._atm_ahead = False
        self._pinned = {}
        self._flip = {}
        self._copy_stream = None
        self._act_dev = None
        self._act_slot = 0
        self._out_ready = None

    def _host_buffers(self, tensors):
        """Two sets of pinned buffers alternate, so the tensors handed out at step t stay valid until step t+2
        (callers that keep observations longer — e.g. a replay buffer — copy them, as they do with the reference's
        arrays)."""
        key = tuple((tuple(t.shape), t.dtype) for t in tensors)
        sets = 3 if self.lookahead else 2
        if key not in self._pinned:
            self._pinned[key] = [[torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in tensors] for _ in range(sets)]
            self._flip[key] = 0
        self._flip[key] = (self._flip[key] + 1) % sets
        return self._pinned[key][self._flip[key]]

    def _to_host(self, *tensors):
        """Asynchronous device->pinned-host copies on the current stream, one stream synchronisation."""
        bufs = self._host_buffers(tensors)
        for p_, t in zip(bufs, tensors):
            p_.copy_(t, non_blocking=True)
        torch.cuda.current_stream(self._env.device).synchronize()
        return bufs

    def _upload(self, action):
        """Action -> device on the copy stream; returns (device tensor, event to wait for or None)."""
        dev = self._env.device
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(dev)
        a = torch.as_tensor(action)
        if a.device.type != "cpu":
            return a, None
        a = a.to(torch.float32)
        if self._act_dev is None or self._act_dev[0].shape != a.shape:
            self._act_dev = [torch.empty(a.shape, dtype=torch.float32, device=dev) for _ in range(2)]
        self._act_slot ^= 1
        a_dev = self._act_dev[self._act_slot]              # the other buffer may still be read by the last command update
        with torch.cuda.stream(self._copy_stream):
            a_dev.copy_(a, non_blocking=True)
            ready = self._copy_stream.record_event()
        return a_dev, ready

    def _download_hook(self, out):
        """Callback for the point of the stream where obs / reward / Strehl are final: copies them to pinned host
        buffers on the copy stream and leaves the completion event in `out`."""
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(self._env.device)
        main = torch.cuda.current_stream(self._env.device)

        def after_observe(obs, reward, strehl):
            seen = main.record_event()
            self._copy_stream.wait_event(seen)
            tensors = (obs, reward, strehl)
            bufs = self._host_buffers(tensors)
            with torch.cuda.stream(self._copy_stream):
                for p_, t in zip(bufs, tensors):
                    p_.copy_(t, non_blocking=True)
                out["ready"] = self._copy_stream.record_event()
            out["bufs"], out["keep"] = bufs, tensors
        return after_observe

    def _step_pipelined(self, i, action):
        """Host tensors in / out with the copies off the critical path: the action goes up on a copy stream while
        the atmosphere and the WFS of this frame run (the command update waits for it), and the observation comes down
        on the copy stream while the command update and the next DM surface are computed."""
        a_dev, ready = self._upload(action)
        out = {}
        self._env._step_views(i, a_dev, action_ready=ready, after_observe=self._download_hook(out))
        out["ready"].synchronize()
        return out["bufs"]

    def _step_lookahead(self, i, action):
        """Stream order per call:  command(t), DM surface(t), WFS + reconstruction(t+1) -> download, atmosphere(t+2).
        The atmosphere of the frame after next depends on nothing the host decides, so it fills the time the host
        needs to turn obs(t+1) into action(t+1) and upload it."""
        env = self._env
        if self._ahead is None:                            # first step after a reset: measure this frame now
            self._ahead = {}
            env._measure_frame(i, self._download_hook(self._ahead), atmosphere_done=self._atm_ahead)
            env.atm.prefetch() or env.atm.update()
            self._atm_ahead = True
        cur = self._ahead
        a_dev, ready = self._upload(action)
        env._apply_command(a_dev, ready)
        # the next observe overwrites the output buffers: it must not start before the download of the frame measured
        # ahead has read them (the upload event orders this only when the action comes from the host)
        torch.cuda.current_stream(env.device).wait_event(cur["ready"])
        self._ahead = {}
        env._measure_frame(None if i is None else i + 1, self._download_hook(self._ahead), atmosphere_done=True)
        env.atm.prefetch() or env.atm.update()      # frame t+2: on the side stream when the batch is large enough
        cur["ready"].synchronize()
        if ready is not None:
            ready.synchronize()            # the caller may reuse its action buffer as soon as step returns
        return cur["bufs"]

    def reset_envs(self, env_ids, seed):
        """OOPAO.reset_envs of the wrapped environment (not in lookahead mode: its next observation is already measured)."""
        if self.lookahead:
            raise NotImplementedError("reset_envs with TorchWrapper(lookahead=True): the next observation has already been "
                                      "measured from the current episodes")
        return self._env.reset_envs(env_ids, seed)

    def flush(self):
        """Drops the frame measured ahead (lookahead mode): the next step measures again from the current state (the
        atmosphere stays one update ahead)."""
        self._ahead = None

    @staticmethod
    def _split(out):
        """(obs, frame or None, reward, strehl, done, info) from a 5-tuple (Razor environment, OOPAOEnvRazor.py:514) or a
        6-tuple with the WFS camera frame in second place (papyrus environment, OOPAOEnv.py:536)."""
        if len(out) == 6:
            return out
        obs, reward, strehl, done, info = out
        return obs, None, reward, strehl, done, info

    def _bare_step_env(self):
        """True when self._env IS an environment whose step can be taken apart (_step_views) — not a wrapper around one
        (TimeDelayEnv must see every action) and not one that also returns the camera frame."""
        from ..OOPAOEnv.OOPAOEnvRazor import OOPAO as _Razor
        return isinstance(self._env, _Razor) and not getattr(self._env, "returns_frame", False)

    def step(self, i, action):
        """util_simple.py:209-213: same arity as the wrapped environment's step (the camera frame, when the environment
        returns one, stays second)."""
        dev = self._env.device
        if not self.host_io:
            a = torch.as_tensor(action)
            if a.device != dev:
                a = a.to(dev, dtype=torch.float32, non_blocking=True)
            obs, frame, reward, strehl, done, info = self._split(self._env.step(i, a))
            info = [(k, v) for k, v in info.items()]
            return (obs, reward, strehl, done, info) if frame is None else (obs, frame, reward, strehl, done, info)
        # small batches are launch-bound: the extra stream / event traffic of the pipelined path costs more than the
        # copies it hides
        big = self._env.n_envs * self._env.nActuator ** 2 >= 65536
        bare = self._bare_step_env()
        frame_h = None
        if self.lookahead and bare:
            obs_h, reward_h, strehl_h = self._step_lookahead(i, action)
        elif big and bare:
            obs_h, reward_h, strehl_h = self._step_pipelined(i, action)
        else:                                           # e.g. an env wrapped in TimeDelayEnv goes through its own step()
            a = torch.as_tensor(action)
            if a.device != dev:
                a = a.to(dev, dtype=torch.float32, non_blocking=True)
            obs, frame, reward, strehl, done, info = self._split(self._env.step(i, a))
            if frame is None:
                obs_h, reward_h, strehl_h = self._to_host(obs, reward, strehl)
            else:
                obs_h, reward_h, strehl_h, frame_h = self._to_host(obs, reward, strehl, frame)
        if self._env.n_envs == 1:
            reward_h, strehl_h = float(reward_h), float(strehl_h)
        info = [("strehl", torch.as_tensor(strehl_h, dtype=torch.float32))]
        if frame_h is not None:
            return obs_h, frame_h, reward_h, strehl_h, False, info
        return obs_h, reward_h, strehl_h, False, info

    def reset_soft(self):
        self._ahead = None
        self._atm_ahead = False            # episode boundary: the caller has just drawn new screens (or accepts a skipped frame)
        obs = self._env.reset_soft()
        return self._to_host(obs)[0] if self.host_io else obs


class ReplaySample:
    """util_simple.py:130-161."""

    def __init__(self, states, actions, rewards, next_states):
        self.states, self.actions, self.rewards, self.next_states = states, actions, rewards, next_states

    def state(self):
        return self.states

    def action(self):
        return self.actions

    def reward(self):
        return self.rewards

    def next_state(self):
        return self.next_states

    def __len__(self):
        return len(self.states)

    def to(self, device):
        self.states, self.actions = self.states.to(device), self.actions.to(device)
        self.rewards, self.next_states = self.rewards.to(device), self.next_states.to(device)
        return self


class EfficientExperienceReplay:
    """util_simple.py:55-128 with the storage on `device` and `n_envs` environments stepping in lock-step.

    Rows are appended time-major: one `append` call stores the transitions of all environments of a step in
    `n_envs` consecutive rows, so an episode of `max_ts` steps is a block of `max_ts * n_envs` rows and the
    trajectory of environment b inside it has stride `n_envs`.  `sample_contiguous` draws windows that stay inside
    one (episode, environment) trajectory; with n_envs == 1 the layout, the index arithmetic and the random-number
    consumption are the reference's (:103-111)."""

    def __init__(self, state_shape, action_shape, max_size=100000, device="cpu", n_envs=1):
        self.max_size = max_size
        self.n_envs = int(n_envs)
        self.device = torch.device(device)
        self.states = torch.empty((max_size, *state_shape), device=self.device)
        self.next_states = torch.empty((max_size, *state_shape), device=self.device)
        self.actions = torch.empty((max_size, *action_shape), device=self.device)
        self.rewards = torch.empty((max_size, 1), device=self.device)
        self.len = 0

    def add(self, replay):
        """:68-81."""
        n = len(replay)
        sl = slice(self.len, self.len + n)
        self.states[sl], self.next_states[sl] = replay.state()[:n], replay.next_state()[:n]
        self.actions[sl], self.rewards[sl] = replay.action()[:n], replay.reward()[:n]
        self.len += n

    def __add__(self, replay):
        self.add(replay)
        return self

    def append(self, obs, action, reward, next_obs, done=False):
        """:87-99; with n_envs > 1 the arguments carry a leading [n_envs] axis."""
        if not torch.is_tensor(obs):
            raise TypeError("should be torch")
        B = self.n_envs
        if self.len + B > self.max_size:
            raise IndexError(f"replay is full ({self.max_size} transitions)")
        if B == 1:
            i = self.len
            self.states[i], self.next_states[i], self.actions[i] = obs, next_obs, action
            self.rewards[i] = reward
        else:
            sl = slice(self.len, self.len + B)
            self.states[sl], self.next_states[sl], self.actions[sl] = obs, next_obs, action
            self.rewards[sl] = torch.as_tensor(reward, device=self.device).reshape(B, 1)
        self.len += B

    def sample_contiguous(self, horizon, max_ts, batch_size=32):
        B = self.n_envs
        start = torch.randint(0, max_ts - (horizon + 1), size=(batch_size,))
        traj = torch.randint(0, len(self) // max_ts, size=(batch_size,))          # (episode, environment) pairs
        first = (traj // B) * (max_ts * B) + (traj % B) + start * B
        indices = (first[:, None] + torch.arange(horizon + 1)[None, :] * B).reshape(-1).to(self.device)
        return ReplaySample(self.states[indices], self.actions[indices], self.rewards[indices], self.next_states[indices])

    def sample(self, size=512):
        inds = torch.randperm(self.len, device=self.device)[:size]
        return ReplaySample(self.states[inds], self.actions[inds], self.rewards[inds], self.next_states[inds])

    def state(self):
        return self.states[:self.len]

    def next_state(self):
        return self.next_states[:self.len]

    def action(self):
        return self.actions[:self.len]

    def reward(self):
        return self.rewards[:self.len]

    def __len__(self):
        return self.len

    def clear(self):
        self.len = 0


def get_n_params(model):
    """util_simple.py:217-224."""
    return sum(p.numel() for p in model.parameters())
