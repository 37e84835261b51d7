from .env_runner import EnvRunner, RunnerWrapper
from .frame_stacks import DeviceFrameStackPacker, FrameStackPacker, FrameStacks
from .onpolicy import (TransformInteractions, IterateWithMinibatches, gather_minibatch,
                       ppo_runner_wrap, make_ppo_runner)
from .summary import PeriodicSummaries
from .synthetic import SyntheticRolloutRunner, SyntheticEnv, make_frame_stack_rollout, make_rollout
from .trajectory_transforms import GAE, MergeTimeBatch, NormalizeAdvantages, Take
