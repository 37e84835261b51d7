"""derl_b200 — B200-native (sm_100a) PPO rollout-processing / update data path behind
mknbv/derl's Python API: GAE -> minibatch gather -> fused PPO loss, rollout resident in HBM.

Importing this package loads libderl_b200.so (build it with `python __graft_entry__.py`);
there is no CPU fallback — without the library the import fails, without an sm_100 GPU
every op raises.
"""
from . import summary
from .alg import (A2C, A2CLoss, Alg, GraphedTrainer, Loss, PPO, PPOLoss, Trainer, r_squared,
                  total_norm)
from .anneal import AnnealingVariable, LinearAnneal
from .models import MLP, MuJoCoModel, NatureCNNBase, NatureCNNModel, make_model, orthogonal_init
from .policies import ActorCriticPolicy, Policy
from .runners import (DeviceFrameStackPacker, EnvRunner, FrameStackPacker, FrameStacks, GAE,
                      IterateWithMinibatches, MergeTimeBatch, NormalizeAdvantages,
                      PeriodicSummaries, RunnerWrapper, SyntheticRolloutRunner, Take, TransformInteractions, make_frame_stack_rollout,
                      make_ppo_runner, make_rollout, ppo_runner_wrap)
