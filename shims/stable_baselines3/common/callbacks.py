"""Name shim: ``from stable_baselines3.common.callbacks import CheckpointCallback`` (examples/train.py:7), and the
rest of SB3's callback surface that is built here."""
from mobrob_b200.callbacks import (  # noqa: F401
    BaseCallback,
    CallbackList,
    CheckpointCallback,
    EvalCallback,
    EventCallback,
    StopTrainingOnRewardThreshold,
)
