"""dexterous_rl_manipulation_b200 -- B200-native batched simulator for the hot path of
I2S9/dexterous-rl-manipulation (stepping many independent DexterousManipulationEnv instances).

Public face: ``BatchedManipulationEnv`` (drop-in for the reference env object),
``CurriculumConfig`` (field-compatible config), the label / counter constants of the C ABI
(include/dexsim.h) and the env-sharding helpers in ``distributed``.
Importing the package loads libdexsim_b200.so and raises if it is missing: no CPU fallback.
"""
from . import _lib
from ._lib import (CNT_EPISODES, CNT_LABEL_METRICS, CNT_LABEL_TAXONOMY, CNT_SUCCESSES, CNT_SUM_FINAL_CONTACTS,
                   CNT_SUM_STEPS, CNT_SUM_STEPS_SQ, CNT_VAR_TIES, LABEL_NONE, LABELS_METRICS, LABELS_TAXONOMY,
                   NCOUNTERS, DexsimError, classify_counts, classify_summary)
from .config import CurriculumConfig, group_from_config, group_table

import sys as _sys

# Fail loudly at import time when the CUDA extension is absent or stale -- except for the one command whose job is
# to produce it (`python -m dexterous_rl_manipulation_b200.build` imports this package before running build.py).
_argv = list(getattr(_sys, "orig_argv", []))
if not ("-m" in _argv and __name__ + ".build" in _argv):
    _lib.lib()

from .env import BatchedManipulationEnv, Box  # noqa: E402
from .policy import MlpPolicy  # noqa: E402
from . import distributed  # noqa: E402
from .curriculum import BatchedCurriculumDriver, CurriculumScheduler  # noqa: E402
from . import evaluation  # noqa: E402
from . import training  # noqa: E402
from .training import run_episodes_batched  # noqa: E402

DexterousManipulationEnv = BatchedManipulationEnv   # the reference's class name, for drop-in imports

__all__ = [
    "BatchedManipulationEnv", "DexterousManipulationEnv", "Box", "MlpPolicy", "CurriculumConfig", "group_from_config",
    "group_table", "classify_summary", "classify_counts", "run_episodes_batched", "evaluation", "training", "BatchedCurriculumDriver", "CurriculumScheduler", "DexsimError", "distributed", "LABELS_METRICS", "LABELS_TAXONOMY",
    "LABEL_NONE", "NCOUNTERS", "CNT_EPISODES", "CNT_SUCCESSES", "CNT_SUM_STEPS", "CNT_SUM_FINAL_CONTACTS",
    "CNT_LABEL_METRICS", "CNT_LABEL_TAXONOMY", "CNT_VAR_TIES", "CNT_SUM_STEPS_SQ",
]
