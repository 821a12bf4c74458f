"""mobrob_b200 -- B200-native goal-conditioned PPO hot path of ZikangXiong/mobrob.

Public surface mirrors the reference package (src/mobrob/__init__.py:1-4): ``get_env`` and
``load_policy``; plus ``GpuVecEnv`` / ``PPO`` / ``PPOCtrl`` for the batched path and SB3's ``evaluate_policy``.
"""
__all__ = ["get_env", "load_policy", "GpuVecEnv", "PPO", "PPOCtrl", "evaluate_policy"]


def __getattr__(name):
    if name == "evaluate_policy":
        from .evaluation import evaluate_policy
        return evaluate_policy
    if name == "GpuVecEnv":
        from .vec_env import GpuVecEnv
        return GpuVecEnv
    if name == "PPO":
        from .ppo import PPO
        return PPO
    if name == "PPOCtrl":
        from .rl_control.ppo import PPOCtrl
        return PPOCtrl
    if name == "get_env":
        from .envs.wrapper import get_env
        return get_env
    if name == "load_policy":
        from .utils import load_policy
        return load_policy
    raise AttributeError(name)
