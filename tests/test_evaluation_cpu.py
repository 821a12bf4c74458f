"""evaluate_policy / EvalCallback host logic without a GPU: the device records' assembly into SB3's order, the step
bound, the shims, and the step-event replay of CallbackList and EvalCallback."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mobrob_b200 import callbacks as cb_mod  # noqa: E402
from mobrob_b200 import evaluation  # noqa: E402


def _sb3_loop(done, ret, n_eval_episodes):
    """SB3 2.0.0 evaluate_policy's loop over a scripted done stream done[t, i] (Monitor return ret[t, i] where done):
    the appended (reward, length-like tag) pairs and the number of steps taken."""
    T, n = done.shape
    counts = np.zeros(n, int)
    targets = np.array([(n_eval_episodes + i) // n for i in range(n)], int)
    out, t = [], 0
    while (counts < targets).any():
        for i in range(n):
            if counts[i] < targets[i] and done[t, i]:
                out.append((ret[t, i], t, i))
                counts[i] += 1
        t += 1
    return out, t


def _device_records(done, ret, n_eval_episodes):
    """What mr_evaluate writes: env i's first c_i episodes in slots off_i .. off_i + c_i - 1, with the ending step."""
    T, n = done.shape
    targets = evaluation.episode_targets(n_eval_episodes, n)
    offsets = np.concatenate([[0], np.cumsum(targets)[:-1]])
    ep_r = np.full(n_eval_episodes, np.nan)
    ep_t = np.full(n_eval_episodes, -1, np.int64)
    ep_env = np.full(n_eval_episodes, -1, np.int64)
    steps = 0
    for i in range(n):
        ends = np.nonzero(done[:, i])[0][:targets[i]]
        assert len(ends) == targets[i]
        ep_r[offsets[i]:offsets[i] + targets[i]] = ret[ends, i]
        ep_t[offsets[i]:offsets[i] + targets[i]] = ends
        ep_env[offsets[i]:offsets[i] + targets[i]] = i
        if len(ends):
            steps = max(steps, int(ends[-1]) + 1)
    return ep_r, ep_t, ep_env, steps


@pytest.mark.parametrize("n_envs,n_eval_episodes", [(8, 3), (8, 8), (7, 23), (5, 40), (1, 4), (16, 0), (96, 250)])
def test_record_order_matches_sb3_loop(n_envs, n_eval_episodes):
    rng = np.random.default_rng(n_envs * 1000 + n_eval_episodes)
    T = 400
    done = rng.random((T, n_envs)) < 0.15
    ret = rng.standard_normal((T, n_envs))
    expected, sb3_steps = _sb3_loop(done, ret, n_eval_episodes)
    ep_r, ep_t, ep_env, steps = _device_records(done, ret, n_eval_episodes)
    # the closed-form slot offsets of the kernel
    targets = evaluation.episode_targets(n_eval_episodes, n_envs)
    assert targets.sum() == n_eval_episodes
    E, N = n_eval_episodes, n_envs
    q, r = divmod(E, N)
    assert [q * i + max(0, i - (N - r)) for i in range(N)] == list(np.concatenate([[0], np.cumsum(targets)[:-1]]))
    order = evaluation.record_order(ep_t, n_envs, n_eval_episodes)
    got = list(zip(ep_r[order], ep_t[order], ep_env[order]))
    assert got == expected
    assert steps == sb3_steps


def test_targets_below_and_above_env_count():
    assert list(evaluation.episode_targets(3, 8)) == [0, 0, 0, 0, 0, 1, 1, 1]
    assert list(evaluation.episode_targets(10, 4)) == [2, 2, 3, 3]


class _ScriptedVecEnv:
    """A VecEnv whose env i finishes an episode every period[i] steps (reward 1 per step); no Monitor infos."""

    def __init__(self, periods, time_limit=None):
        self.periods = np.asarray(periods)
        self.num_envs = len(periods)
        self.time_limit = time_limit
        self.t = 0
        self.resets = 0

    def reset(self):
        self.t = 0
        self.resets += 1
        return np.zeros((self.num_envs, 1), np.float32)

    def step(self, actions):
        self.t += 1
        dones = self.t % self.periods == 0
        return np.zeros((self.num_envs, 1), np.float32), np.ones(self.num_envs), dones, [{} for _ in range(self.num_envs)]


class _ConstModel:
    seed = 0

    def predict(self, obs, state=None, episode_start=None, deterministic=False):
        return np.zeros((len(obs), 2), np.float32), state


def test_max_steps_required_without_time_limit():
    env = _ScriptedVecEnv([3, 5], time_limit=None)
    with pytest.raises(ValueError, match="max_steps"):
        evaluation.evaluate_policy(_ConstModel(), env, n_eval_episodes=4, warn=False)
    assert env.resets == 0
    env.time_limit = 0
    with pytest.raises(ValueError, match="max_steps"):
        evaluation.resolve_max_steps(env, 4, None)
    # with a time limit: ceil(n_eval_episodes / n_envs) episodes of at most time_limit steps each
    env.time_limit = 100
    assert evaluation.resolve_max_steps(env, 5, None) == 300
    assert evaluation.resolve_max_steps(env, 5, 7) == 7


def test_generic_loop_results_and_step_bound():
    env = _ScriptedVecEnv([3, 5], time_limit=None)
    with pytest.warns(UserWarning, match="Monitor"):
        rewards, lengths = evaluation.evaluate_policy(_ConstModel(), env, n_eval_episodes=5, max_steps=100,
                                                      return_episode_rewards=True)
    # env 0 counts 2 episodes (steps 3, 6), env 1 counts 3 (steps 5, 10, 15): (step, env) order
    assert lengths == [3, 5, 3, 5, 5] and rewards == [3.0, 5.0, 3.0, 5.0, 5.0]
    assert env.t == 15
    with pytest.raises(RuntimeError, match="max_steps"):
        evaluation.evaluate_policy(_ConstModel(), env, n_eval_episodes=5, max_steps=12, warn=False)
    assert env.t == 12
    mean, std = evaluation.evaluate_policy(_ConstModel(), env, n_eval_episodes=5, max_steps=100, warn=False)
    assert mean == pytest.approx(4.2) and std == pytest.approx(np.std([3, 5, 3, 5, 5]))
    with pytest.raises(AssertionError):
        evaluation.evaluate_policy(_ConstModel(), env, n_eval_episodes=5, max_steps=100, warn=False, reward_threshold=5)


def test_generic_loop_passes_locals_to_callback():
    env = _ScriptedVecEnv([2, 4], time_limit=4)
    seen = []
    evaluation.evaluate_policy(_ConstModel(), env, n_eval_episodes=2, warn=False,
                               callback=lambda l, g: seen.append((env.t, l["i"], bool(l["done"]))))
    # one call per env per step while the env is short of its target (env 0: 1 episode, env 1: 1 episode)
    assert seen == [(1, 0, False), (1, 1, False), (2, 0, True), (2, 1, False), (3, 1, False), (4, 1, True)]


def test_shims_resolve():
    code = "\n".join([
        "import sys", f"sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'shims')!r}]",
        "from stable_baselines3.common.evaluation import evaluate_policy",
        "from stable_baselines3.common.callbacks import (BaseCallback, CallbackList, CheckpointCallback, EvalCallback,",
        "    EventCallback, StopTrainingOnRewardThreshold)",
        "import mobrob_b200, mobrob_b200.callbacks as c, mobrob_b200.evaluation as e",
        "assert evaluate_policy is e.evaluate_policy is mobrob_b200.evaluate_policy",
        "assert EvalCallback is c.EvalCallback and CallbackList is c.CallbackList",
        "assert StopTrainingOnRewardThreshold is c.StopTrainingOnRewardThreshold and EventCallback is c.EventCallback",
        "print('ok')"])
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


class _FakeModel:
    def __init__(self, n_envs=2):
        self.n_envs, self.num_timesteps, self.saved = n_envs, 0, []
        self.logger = _FakeLogger()

    def _world_size(self):
        return 1

    def _is_rank0(self):
        return True

    def save(self, path):
        self.saved.append((os.path.basename(path), self.num_timesteps))


class _FakeLogger:
    def __init__(self):
        self.records, self.dumps = {}, []

    def record(self, key, value, exclude=None):
        self.records[key] = value

    def dump(self, step=0):
        self.dumps.append((step, dict(self.records)))
        self.records = {}


class _Probe(cb_mod.BaseCallback):
    def __init__(self, name, log, stop_at=None):
        super().__init__()
        self.name, self.log, self.stop_at = name, log, stop_at

    def _on_step(self):
        self.log.append((self.name, self.n_calls, self.num_timesteps, self.model.num_timesteps))
        return self.stop_at is None or self.n_calls < self.stop_at


def test_callback_list_replays_steps_interleaved_and_stops_at_first_false(tmp_path):
    m = _FakeModel()
    log = []
    ckpt = cb_mod.CheckpointCallback(save_freq=3, save_path=str(tmp_path), name_prefix="ck")
    lst = cb_mod.CallbackList([_Probe("a", log), ckpt, _Probe("b", log, stop_at=6)])
    lst.init_callback(m)
    lst.on_training_start({}, {})
    m.num_timesteps += 4 * m.n_envs
    assert lst.on_rollout_steps(4) is True
    assert m.num_timesteps == 8
    m.num_timesteps += 4 * m.n_envs
    assert lst.on_rollout_steps(4) is False        # b returns False on its 6th call
    assert m.num_timesteps == 16                   # restored to the end of the rollout
    # per step: a then b (children in list order), each with the step's own num_timesteps, on the model too
    exp = []
    for k in range(1, 7):
        exp += [("a", k, 2 * k, 2 * k), ("b", k, 2 * k, 2 * k)]
    assert log == exp
    assert m.saved == [("ck_6_steps.zip", 6), ("ck_12_steps.zip", 12)]
    assert lst.n_calls == 6 and ckpt.n_calls == 6


class _EpisodeEnv:
    """Eval env stand-in: every env ends an episode each step with reward = the value the model reports."""

    num_envs = 2
    time_limit = 1

    def __init__(self, model):
        self.model = model

    def reset(self):
        return np.zeros((2, 1), np.float32)

    def step(self, actions):
        r = np.full(2, float(self.model.quality))
        infos = [{"episode": {"r": r[0], "l": 1}, "is_success": True} for _ in range(2)]
        return np.zeros((2, 1), np.float32), r, np.ones(2, bool), infos


def test_eval_callback_logs_saves_best_and_stops(tmp_path, capsys):
    m = _FakeModel()
    m.quality = 1.0
    m.predict = _ConstModel().predict
    env = _EpisodeEnv(m)
    stop = cb_mod.StopTrainingOnRewardThreshold(reward_threshold=2.5, verbose=1)
    ev = cb_mod.EvalCallback(env, callback_on_new_best=stop, n_eval_episodes=4, eval_freq=3,
                             log_path=str(tmp_path / "logs"), best_model_save_path=str(tmp_path / "best"), warn=False)
    lst = cb_mod.CallbackList([ev])
    lst.init_callback(m)
    lst.on_training_start({}, {})
    qualities = iter([3.0, 2.0])
    keep = True
    rollouts = 0
    while keep and rollouts < 10:
        m.num_timesteps += 4 * m.n_envs
        rollouts += 1
        # the model's parameters only change between rollouts
        m.quality = next(qualities) if rollouts > 1 else 1.0
        keep = lst.on_rollout_steps(4)
    # evaluations at step events 3 and 6: num_timesteps 6 and 12; the second is a new best above the threshold
    assert not keep and rollouts == 2
    z = np.load(tmp_path / "logs" / "evaluations.npz")
    assert list(z["timesteps"]) == [6, 12]
    assert z["results"].tolist() == [[1.0] * 4, [3.0] * 4] and z["ep_lengths"].tolist() == [[1] * 4] * 2
    assert z["successes"].tolist() == [[True] * 4] * 2
    assert m.saved == [("best_model", 6), ("best_model", 12)]
    assert ev.best_mean_reward == 3.0 and ev.last_mean_reward == 3.0
    assert [d[0] for d in m.logger.dumps] == [6, 12]
    assert m.logger.dumps[1][1]["eval/mean_reward"] == 3.0 and m.logger.dumps[1][1]["eval/success_rate"] == 1.0
    out = capsys.readouterr().out
    assert "Eval num_timesteps=12, episode_reward=3.00 +/- 0.00" in out and "New best mean reward!" in out
    assert "Episode length: 1.00 +/- 0.00" in out and "Stopping training" in out


def test_eval_callback_refuses_several_ranks():
    m = _FakeModel()
    m._world_size = lambda: 2
    ev = cb_mod.EvalCallback(_EpisodeEnv(m), eval_freq=1)
    with pytest.raises(NotImplementedError):
        ev.init_callback(m)
