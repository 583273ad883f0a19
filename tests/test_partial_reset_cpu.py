"""Per-environment episode resets without a GPU: the bookkeeping of GymnasiumVectorSH (who truncates and resets at each
call, with and without staggered episodes, ignored actions, cleared history / FIFO rows, zero reward at the reset step) on
a stub environment, and OOPAO.reset_envs on the CPU stand-in of the library (unlisted rows of every buffer untouched,
listed ones redrawn with a flat mirror)."""
import types

import numpy as np
import pytest
import torch

import fake_backend_partial_reset
from oracle.golden_configs import CONFIGS
from parity_util import build_env
from rlao_b200.OOPAOEnv.gymnasium_api import GymnasiumVectorSH


class StubEnv:
    """The part of OOPAO the vector wrapper uses; obs = delayed action + 1, Strehl = 0.5 + env index / 100."""

    def __init__(self, B, nA=3):
        self.n_envs, self.nActuator, self.device = B, nA, torch.device("cpu")
        self.dm = types.SimpleNamespace(nValidAct=999)
        self.resets, self.seen = [], []

    def reset_envs(self, ids, seed):
        ids = [int(i) for i in np.asarray(ids)]
        self.resets.append((ids, seed))
        return torch.as_tensor(ids, dtype=torch.int32)

    def _step_views(self, i, delayed):
        self.seen.append(delayed.clone())
        strehl = 0.5 + torch.arange(self.n_envs, dtype=torch.float32) / 100
        return delayed + 1.0, -strehl, strehl, False, {}


def run_schedule(B, L, stagger, calls):
    env = StubEnv(B)
    vec = GymnasiumVectorSH(env, n_history=4, delay=1, episode_length=L, stagger_episodes=stagger)
    vec._steps = vec._start_steps()                           # (a full reset needs the real objects: start from the counters)
    trunc, auto = [], []
    for t in range(calls):
        _, reward, terminated, truncated, info = vec.step(torch.zeros((B, 3, 3)))
        assert not terminated.any()
        assert not truncated[info["autoreset"]].any()
        assert (reward.numpy()[info["autoreset"]] == 0).all()
        trunc.append(np.nonzero(truncated)[0].tolist())
        auto.append(np.nonzero(info["autoreset"])[0].tolist())
    return env, trunc, auto


def test_truncation_and_autoreset_lock_step():
    env, trunc, auto = run_schedule(4, 3, False, 8)
    assert trunc == [[], [], [0, 1, 2, 3], [], [], [], [0, 1, 2, 3], []]
    assert auto == [[], [], [], [0, 1, 2, 3], [], [], [], [0, 1, 2, 3]]
    assert [r[0] for r in env.resets] == [[0, 1, 2, 3], [0, 1, 2, 3]]


def test_staggered_episodes_spread_the_resets():
    B, L = 4, 8                                               # environment e starts at step e * L // B = 0, 2, 4, 6
    env, trunc, auto = run_schedule(B, L, True, 20)
    assert trunc[:9] == [[], [3], [], [2], [], [1], [], [0], []]
    assert auto[:9] == [[], [], [3], [], [2], [], [1], [], [0]]
    assert trunc[10] == [3] and auto[11] == [3]               # a full episode (L steps) after its reset call
    assert [r[0] for r in env.resets[:4]] == [[3], [2], [1], [0]]
    assert all(len(t) <= 1 for t in trunc)                    # never more than one environment at a time


def test_no_truncation_without_episode_length():
    env = StubEnv(3)
    vec = GymnasiumVectorSH(env, episode_length=None, stagger_episodes=True)
    for _ in range(5):
        _, _, terminated, truncated, info = vec.step(torch.zeros((3, 3, 3)))
        assert not truncated.any() and not terminated.any() and not info["autoreset"].any()
    assert env.resets == []


def test_reset_step_ignores_the_action_and_clears_history_and_fifo():
    B, d = 3, 2
    env = StubEnv(B)
    vec = GymnasiumVectorSH(env, n_history=4, delay=d, episode_length=4, stagger_episodes=True)   # starts 0, 1, 2
    vec._steps = vec._start_steps()
    acts = [torch.full((B, 3, 3), float(t + 1)) for t in range(8)]
    outs = [vec.step(a) for a in acts]
    # environment 2 truncates at call 1 (index 1) and resets at call 2
    assert outs[1][3].tolist() == [False, False, True] and outs[2][4]["autoreset"].tolist() == [False, False, True]
    seen = torch.stack(env.seen)                              # [call, B, 3, 3] actions the step applied
    for t in range(4):                                        # environment 0 before its reset: the action of d calls earlier
        assert torch.equal(seen[t, 0], torch.full((3, 3), float(t + 1 - d)) if t >= d else torch.zeros(3, 3))
    # environment 2: FIFO cleared and the reset call's own action ignored -> zero for d + 1 calls, then the next action
    assert (seen[2:5, 2] == 0).all() and torch.equal(seen[5, 2], torch.full((3, 3), 4.0))
    obs, reward = outs[2][0], outs[2][1]
    assert reward[2] == 0 and reward[0] == pytest.approx(0.5) and reward[1] == pytest.approx(0.51)
    assert (obs[2, 1:] == 0).all() and torch.equal(obs[2, 0], torch.ones(3, 3))        # history of the new episode only
    assert torch.equal(obs[0, 1], outs[1][0][0, 0])                                       # the others keep theirs


def test_seeded_resets_are_reproducible_and_masked_reset():
    def run(seed):
        env = StubEnv(4)
        vec = GymnasiumVectorSH(env, episode_length=2, stagger_episodes=True)
        vec._rng = np.random.RandomState(seed)
        vec._steps = vec._start_steps()
        for _ in range(6):
            vec.step(torch.zeros((4, 3, 3)))
        obs, _ = vec.reset(options={"reset_mask": np.array([True, False, False, True])})
        return env.resets, vec
    r1, vec = run(5)
    r2, _ = run(5)
    assert r1 == r2 and r1[-1][0] == [0, 3]
    assert len({s for _, s in r1}) == len(r1)
    assert vec._steps[0] == 0 and vec._steps[3] == 0
    with pytest.raises(ValueError):
        vec.reset(options={"reset_mask": np.array([True, False])})


# ---- OOPAO.reset_envs on the CPU stand-in ---------------------------------------------------------------------------------
@pytest.fixture
def fake(monkeypatch):
    return fake_backend_partial_reset.install(monkeypatch)


def _snapshot(env):
    a, dm = env.atm, env.dm
    return dict(maps=a._maps.clone(), ext=a._ext.clone(), dm_prev=env._dm_prev.clone(), coefs=dm._coefs.clone(),
                rows=None if dm._rows is None else dm._rows.clone(), opd=a._opd.clone())


@pytest.mark.parametrize("native", [True, False])
def test_reset_envs_touches_only_the_listed_rows(fake, monkeypatch, native):
    monkeypatch.setenv("AOENV_STEP_NATIVE", "1" if native else "0")
    cfg = CONFIGS["tiny"]()
    B, listed, others = 4, [0, 3], [1, 2]
    twin, env = build_env(cfg, n_envs=B, rng="philox", seed=2), build_env(cfg, n_envs=B, rng="philox", seed=2)
    obs_t = obs_e = None
    for i in range(3):
        act = torch.full((B, env.nActuator, env.nActuator), 0.01 * (i + 1))
        obs_t = twin.step(i, act)[0]
        obs_e = env.step(i, act)[0]
    assert torch.equal(obs_t, obs_e)
    before = _snapshot(env)
    idx = env.reset_envs(np.array([3, 0, 3]), seed=11)                      # duplicates and order do not matter
    assert idx.tolist() == listed and env.atm._prefetched
    after = _snapshot(env)
    for k in ("maps", "ext", "dm_prev", "coefs", "rows", "opd"):
        if after[k] is None:
            continue
        ax = {"maps": 2, "ext": 2, "rows": 1}.get(k, 0)
        assert torch.equal(after[k].index_select(ax, torch.tensor(others)), before[k].index_select(ax, torch.tensor(others))), k
    assert (after["dm_prev"][listed] == 0).all() and (after["coefs"][listed] == 0).all()
    if after["rows"] is not None:
        assert (after["rows"][env.dm._slot][listed] == 0).all()
    M, pitch, atm = env.atm._M, env.atm._pitch, env.atm
    for i in range(atm.nLayer):
        oy, ox = atm._org[i]
        win = atm._maps[i, atm._cur[i], :, oy:oy + M, ox:ox + M]
        for e in listed:
            assert not torch.equal(win[e], before["maps"][i, atm._cur[i], e, oy:oy + M, ox:ox + M])
            ext = atm._ext[i, :, e].numpy().view(np.uint64)
            assert fake._unkey(ext[0, 0]) == win[e].min() and fake._unkey(ext[0, 1]) == win[e].max()
            assert fake._unkey(ext[1, 0]) == win[e, 1:-1, 1:-1].min() and fake._unkey(ext[1, 1]) == win[e, 1:-1, 1:-1].max()
            assert int(ext[2, 0]) == (1 << 32) | (oy * pitch + ox)
    for i in range(3, 7):
        act = torch.full((B, env.nActuator, env.nActuator), 0.01 * (i + 1))
        out_t, out_e = twin.step(i, act), env.step(i, act)
        assert torch.equal(out_t[0][others], out_e[0][others]) and torch.equal(out_t[1][others], out_e[1][others])
        assert torch.equal(twin.atm._opd[others], env.atm._opd[others])
        if i == 3:
            assert not torch.equal(out_t[0][listed], out_e[0][listed])
            # first step of the new episode: flat mirror, so the command is this step's action alone
            assert torch.equal(env._dm_prev[listed, :env.dm.nValidAct], torch.full((2, env.dm.nValidAct), np.float32(0.04) * np.float32(1e-6)))
    assert torch.equal(twin._dm_prev[others], env._dm_prev[others])
    assert [ly.events for ly in env.atm._layers] == [ly.events for ly in twin.atm._layers]      # add_row counters unmoved


def test_reset_envs_refusals(fake):
    cfg = CONFIGS["tiny"]()
    ref = build_env(cfg, n_envs=2, rng="reference")
    with pytest.raises(NotImplementedError, match="reference"):
        ref.reset_envs([0], 1)
    env = build_env(cfg, n_envs=2, rng="philox")
    env.atm.xi_log = []
    with pytest.raises(NotImplementedError, match="xi_log"):
        env.reset_envs([0], 1)
    env.atm.xi_log = None
    env.atm.update(OPD=np.zeros((env.tel.resolution, env.tel.resolution)))
    with pytest.raises(NotImplementedError, match="OPD"):
        env.reset_envs([0], 1)
    env.atm.update()
    with pytest.raises(ValueError):
        env.reset_envs([2], 1)
    with pytest.raises(ValueError):
        env.reset_envs(torch.tensor([True, False, True]), 1)
    assert env.reset_envs([], 1).numel() == 0 and not env.atm._prefetched
    from rlao_b200.OOPAOEnv.OOPAOEnv import OOPAO as PyramidEnv
    from rlao_b200.PO4AO.util_simple import TorchWrapper
    with pytest.raises(NotImplementedError, match="Pyramid"):
        PyramidEnv.reset_envs(object.__new__(PyramidEnv), [0], 1)
    with pytest.raises(NotImplementedError, match="lookahead"):
        TorchWrapper(env, lookahead=True).reset_envs([0], 1)
    assert TorchWrapper(env).reset_envs(np.array([False, True]), 3).tolist() == [1]
