"""relearn_b200 -- B200-native rollout/update hot path of edlanglois/relearn.

Host-side mirror of the reference's interfaces for that path over a C-ABI CUDA library
(`include/relearn_b200.h`, built in-tree by `__graft_entry__.build()`).  No CPU fallback exists.
"""
from . import _lib  # noqa: F401
from .envs import (BatchedEnv, CartPole, CartPoleConfig, Chain, LatentStepLimit, MemoryGame, MetaEnv, OneHotBandits, PartitionGame, Successor,  # noqa: F401
                   TrialEpisodeLimit, UniformBernoulliBandits, VisibleStepLimit, build_env)
from .modules import (GruLinear, GruLinearConfig, LstmLinear, LstmLinearConfig, Mlp, MlpConfig, init_gru_linear_params,  # noqa: F401
                      init_lstm_linear_params, init_params, lstm_linear_num_params, num_params)
from .runtime import Context, DeviceBuffer  # noqa: F401
from .simulation import (ActorSpec, HistoryDataBound, TrainParallelConfig, Trajectory, pack_history, rollout, train_device,  # noqa: F401
                         train_serial)
from .logging import DisplayLogger, HistoryLogger, NullLogger, StatsLogger  # noqa: F401

__version__ = "0.1.0"
from .agents import (BetaThompsonSamplingAgent, BetaThompsonSamplingAgentConfig, RandomAgentConfig,  # noqa: F401,E402
                     ResettingMetaAgent, ResettingMetaAgentConfig, TabularQ, TabularQLearningAgentConfig, UCB1Agent,
                     UCB1AgentConfig)
from .torch_agents import (ActorCriticAgent, ActorCriticConfig, Adam, AdamConfig,  # noqa: F401,E402
                           ConjugateGradientOptimizerConfig, DataCollectionSchedule, DqnAgent, DqnConfig,
                           ExplorationRateSchedule, OptimizerStepError, Ppo, PpoConfig, Reinforce, ReinforceConfig,
                           ReplayBuffer, Trpo, TrpoConfig, ValuesOpt,
                           ValuesOptConfig)
from .serialize import load_actor, save_actor  # noqa: F401,E402
