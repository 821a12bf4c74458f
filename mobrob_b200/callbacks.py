"""The [SB3 2.0.0] callback surface: ``CheckpointCallback`` (examples/train.py:36-41), ``EvalCallback``,
``StopTrainingOnRewardThreshold``, ``EventCallback`` and ``CallbackList``.

SB3 calls ``callback.on_step()`` after every ``VecEnv.step``; here a rollout is one kernel launch,
so ``PPO.learn`` reports whole rollouts with ``on_rollout_steps(n)`` and the callback replays the
n step events it would have seen.  A checkpoint that SB3 would write in the middle of a rollout
holds the same policy (parameters only change in ``train``) and gets the same file name
(``{name_prefix}_{num_timesteps}_steps.zip`` with the step's own ``num_timesteps``).  An evaluation
that falls inside a rollout likewise sees the rollout's parameters and that step's ``num_timesteps``.
"""
from __future__ import annotations

import os
import warnings

import numpy as np


class BaseCallback:
    def __init__(self, verbose: int = 0):
        self.verbose = verbose
        self.model = None
        self.n_calls = 0
        self.num_timesteps = 0
        self.locals, self.globals = {}, {}
        self.parent = None

    # -- SB3 protocol ---------------------------------------------------------------------------
    def init_callback(self, model) -> None:
        self.model = model
        self._init_callback()

    def _init_callback(self) -> None:
        pass

    def on_training_start(self, locals_, globals_) -> None:
        self.locals, self.globals = locals_, globals_
        self.num_timesteps = self.model.num_timesteps
        self._on_training_start()

    def _on_training_start(self) -> None:
        pass

    def on_rollout_start(self) -> None:
        pass

    def on_step(self) -> bool:
        self.n_calls += 1
        self.num_timesteps = self.model.num_timesteps
        return self._on_step()

    def _on_step(self) -> bool:
        return True

    def on_rollout_end(self) -> None:
        pass

    def on_training_end(self) -> None:
        pass

    def update_locals(self, locals_) -> None:
        self.locals.update(locals_)
        self.update_child_locals(locals_)

    def update_child_locals(self, locals_) -> None:
        pass

    # -- batched form used by mobrob_b200.PPO.learn ---------------------------------------------------
    def on_rollout_steps(self, n_steps: int) -> bool:
        """n_steps VecEnv steps have just been taken (model.num_timesteps already counts them)."""
        end = self.model.num_timesteps
        per_step = self.model.n_envs * self.model._world_size()
        keep_going = True
        for k in range(n_steps):
            self.n_calls += 1
            self.num_timesteps = end - (n_steps - 1 - k) * per_step
            if self._on_step() is False:
                keep_going = False
        return keep_going


class CheckpointCallback(BaseCallback):
    """Save the model every ``save_freq`` calls of ``env.step()`` (per-env steps), like SB3's."""

    def __init__(self, save_freq: int, save_path: str, name_prefix: str = "rl_model",
                 save_replay_buffer: bool = False, save_vecnormalize: bool = False, verbose: int = 0):
        super().__init__(verbose)
        self.save_freq = max(int(save_freq), 1)
        self.save_path = save_path
        self.name_prefix = name_prefix

    def _init_callback(self) -> None:
        if self.save_path is not None:
            os.makedirs(self.save_path, exist_ok=True)

    def _checkpoint_path(self, checkpoint_type: str = "", extension: str = "") -> str:
        return os.path.join(self.save_path, f"{self.name_prefix}_{checkpoint_type}{self.num_timesteps}_steps.{extension}")

    def _on_step(self) -> bool:
        if self.n_calls % self.save_freq == 0:
            path = self._checkpoint_path(extension="zip")
            if self.model._is_rank0():
                self.model.save(path)
                if self.verbose >= 2:
                    print(f"Saving model checkpoint to {path}")
        return True


def _replay_step_events(callback: BaseCallback, n_steps: int) -> bool:
    """Replay the n_steps ``on_step`` events of a rollout that has just been collected.  During step k the model's
    ``num_timesteps`` is that step's own count, which is what SB3's callbacks read from it (an evaluation or a save in
    the middle of the rollout carries it).  Stops at the first event that returns False, as SB3's
    ``collect_rollouts`` does; the model's count is restored to the end of the rollout afterwards."""
    model = callback.model
    end = model.num_timesteps
    per_step = model.n_envs * model._world_size()
    try:
        for k in range(n_steps):
            model.num_timesteps = end - (n_steps - 1 - k) * per_step
            if callback.on_step() is False:
                return False
        return True
    finally:
        model.num_timesteps = end


class EventCallback(BaseCallback):
    """Base class for callbacks that trigger a child callback on an event (SB3's ``EventCallback``)."""

    def __init__(self, callback: BaseCallback | None = None, verbose: int = 0):
        super().__init__(verbose=verbose)
        self.callback = callback
        if callback is not None:
            self.callback.parent = self

    def init_callback(self, model) -> None:
        super().init_callback(model)
        if self.callback is not None:
            self.callback.init_callback(self.model)

    def _on_training_start(self) -> None:
        if self.callback is not None:
            self.callback.on_training_start(self.locals, self.globals)

    def _on_event(self) -> bool:
        if self.callback is not None:
            return self.callback.on_step()
        return True

    def update_child_locals(self, locals_) -> None:
        if self.callback is not None:
            self.callback.update_locals(locals_)


class CallbackList(BaseCallback):
    """Several callbacks run as one (SB3's ``CallbackList``; ``PPO.learn`` wraps a list in it).  Every child sees every
    step event, children in list order within a step; training stops after a step on which any child returned
    False."""

    def __init__(self, callbacks: list):
        super().__init__()
        assert isinstance(callbacks, list)
        self.callbacks = callbacks

    def _init_callback(self) -> None:
        for callback in self.callbacks:
            callback.init_callback(self.model)

    def _on_training_start(self) -> None:
        for callback in self.callbacks:
            callback.on_training_start(self.locals, self.globals)

    def on_rollout_start(self) -> None:
        for callback in self.callbacks:
            callback.on_rollout_start()

    def _on_step(self) -> bool:
        continue_training = True
        for callback in self.callbacks:
            # every child runs, even after one has asked to stop
            continue_training = callback.on_step() and continue_training
        return continue_training

    def on_rollout_end(self) -> None:
        for callback in self.callbacks:
            callback.on_rollout_end()

    def on_training_end(self) -> None:
        for callback in self.callbacks:
            callback.on_training_end()

    def update_child_locals(self, locals_) -> None:
        for callback in self.callbacks:
            callback.update_locals(locals_)

    def on_rollout_steps(self, n_steps: int) -> bool:
        return _replay_step_events(self, n_steps)


class StopTrainingOnRewardThreshold(BaseCallback):
    """Stop training once the parent ``EvalCallback``'s best mean reward reaches ``reward_threshold`` (use it as
    ``callback_on_new_best``)."""

    def __init__(self, reward_threshold: float, verbose: int = 0):
        super().__init__(verbose=verbose)
        self.reward_threshold = reward_threshold

    def _on_step(self) -> bool:
        assert self.parent is not None, "``StopTrainingOnMinimumReward`` callback must be used with an ``EvalCallback``"
        continue_training = bool(self.parent.best_mean_reward < self.reward_threshold)
        if self.verbose >= 1 and not continue_training:
            print(f"Stopping training because the mean reward {self.parent.best_mean_reward:.2f} "
                  f" is above the threshold {self.reward_threshold}")
        return continue_training


class EvalCallback(EventCallback):
    """Evaluate the policy every ``eval_freq`` step events (calls of ``env.step()``) with ``evaluate_policy``, log the
    results to ``log_path/evaluations.npz``, keep the best model as ``best_model_save_path/best_model.zip`` and run
    ``callback_on_new_best`` / ``callback_after_eval`` (SB3 2.0.0's ``EvalCallback``).  On a ``GpuVecEnv`` the
    evaluation runs on the device; its infos carry no ``is_success``, so no success rate is logged there."""

    def __init__(self, eval_env, callback_on_new_best: BaseCallback | None = None,
                 callback_after_eval: BaseCallback | None = None, n_eval_episodes: int = 5, eval_freq: int = 10000,
                 log_path: str | None = None, best_model_save_path: str | None = None, deterministic: bool = True,
                 render: bool = False, verbose: int = 1, warn: bool = True):
        super().__init__(callback_after_eval, verbose=verbose)
        self.callback_on_new_best = callback_on_new_best
        if self.callback_on_new_best is not None:
            self.callback_on_new_best.parent = self
        self.n_eval_episodes = n_eval_episodes
        self.eval_freq = eval_freq
        self.best_mean_reward = -np.inf
        self.last_mean_reward = -np.inf
        self.deterministic = deterministic
        self.render = render
        self.warn = warn
        self.eval_env = eval_env
        self.best_model_save_path = best_model_save_path
        if log_path is not None:
            log_path = os.path.join(log_path, "evaluations")
        self.log_path = log_path
        self.evaluations_results = []
        self.evaluations_timesteps = []
        self.evaluations_length = []
        self._is_success_buffer = []
        self.evaluations_successes = []

    def _init_callback(self) -> None:
        if self.model._world_size() > 1:
            # each rank would decide on its own whether to stop, and the ranks' collectives would then hang
            raise NotImplementedError("EvalCallback is not available with several torch.distributed ranks")
        training_env = self.model.get_env() if hasattr(self.model, "get_env") else None
        if training_env is not None and not isinstance(training_env, type(self.eval_env)):
            warnings.warn("Training and eval env are not of the same type" f"{training_env} != {self.eval_env}")
        if self.best_model_save_path is not None:
            os.makedirs(self.best_model_save_path, exist_ok=True)
        if self.log_path is not None:
            os.makedirs(os.path.dirname(self.log_path), exist_ok=True)
        if self.callback_on_new_best is not None:
            self.callback_on_new_best.init_callback(self.model)

    def _log_success_callback(self, locals_, globals_) -> None:
        info = locals_["info"]
        if locals_["done"]:
            maybe_is_success = info.get("is_success")
            if maybe_is_success is not None:
                self._is_success_buffer.append(maybe_is_success)

    def _evaluate(self):
        from .evaluation import _is_gpu_vec_env, evaluate_policy

        # a per-step callback would force the host loop; a GpuVecEnv has no is_success to collect anyway
        callback = None if _is_gpu_vec_env(self.eval_env) else self._log_success_callback
        return evaluate_policy(self.model, self.eval_env, n_eval_episodes=self.n_eval_episodes, render=self.render,
                               deterministic=self.deterministic, return_episode_rewards=True, warn=self.warn,
                               callback=callback)

    def _on_step(self) -> bool:
        continue_training = True
        if self.eval_freq > 0 and self.n_calls % self.eval_freq == 0:
            self._is_success_buffer = []
            episode_rewards, episode_lengths = self._evaluate()
            if self.log_path is not None:
                self.evaluations_timesteps.append(self.num_timesteps)
                self.evaluations_results.append(episode_rewards)
                self.evaluations_length.append(episode_lengths)
                kwargs = {}
                if len(self._is_success_buffer) > 0:
                    self.evaluations_successes.append(self._is_success_buffer)
                    kwargs = dict(successes=self.evaluations_successes)
                np.savez(self.log_path, timesteps=self.evaluations_timesteps, results=self.evaluations_results,
                         ep_lengths=self.evaluations_length, **kwargs)
            mean_reward, std_reward = np.mean(episode_rewards), np.std(episode_rewards)
            mean_ep_length, std_ep_length = np.mean(episode_lengths), np.std(episode_lengths)
            self.last_mean_reward = mean_reward
            if self.verbose >= 1:
                print(f"Eval num_timesteps={self.num_timesteps}, episode_reward={mean_reward:.2f} +/- {std_reward:.2f}")
                print(f"Episode length: {mean_ep_length:.2f} +/- {std_ep_length:.2f}")
            logger = self.model.logger
            logger.record("eval/mean_reward", float(mean_reward))
            logger.record("eval/mean_ep_length", mean_ep_length)
            if len(self._is_success_buffer) > 0:
                success_rate = np.mean(self._is_success_buffer)
                if self.verbose >= 1:
                    print(f"Success rate: {100 * success_rate:.2f}%")
                logger.record("eval/success_rate", success_rate)
            logger.record("time/total_timesteps", self.num_timesteps, exclude="tensorboard")
            logger.dump(self.num_timesteps)
            if mean_reward > self.best_mean_reward:
                if self.verbose >= 1:
                    print("New best mean reward!")
                if self.best_model_save_path is not None:
                    self.model.save(os.path.join(self.best_model_save_path, "best_model"))
                self.best_mean_reward = mean_reward
                if self.callback_on_new_best is not None:
                    continue_training = self.callback_on_new_best.on_step()
            if self.callback is not None:
                continue_training = continue_training and self._on_event()
        return continue_training

    def on_rollout_steps(self, n_steps: int) -> bool:
        return _replay_step_events(self, n_steps)
