"""Name shim: ``from stable_baselines3.common.evaluation import evaluate_policy``."""
from mobrob_b200.evaluation import evaluate_policy  # noqa: F401
