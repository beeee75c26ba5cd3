"""B200-native batched simulator for the env.step() hot path of PointTSP / TimedTSP /
ColourMatch (andrewli77/combinatorial-rl-tasks).  See DESIGN.md."""
from .config import ENV_SPECS, TaskSpec  # noqa: F401
from .vec_env import EnvSnapshot, ZoneVecEnv, make_vec_env  # noqa: F401
from .compat import GymEnv, ParallelEnv, TimeoutWrapper, make_fixed_env, make_test_env, make_train_env  # noqa: F401
from .encoder import FusedZoneEnvModel, ZoneEncoder  # noqa: F401
