"""Dumps the widowGo1 training configuration of the reference (WidowGo1RoughCfgPPO, legged_gym/envs/widowGo1/widowGo1_config.py:317-383)
to baseline/widowgo1_train_cfg.json, so that bench.py can construct the reference's own ActorCritic / PPO where
legged_gym (which needs isaacgym) cannot be imported.  Run with a checkout of the original repository:
DWBC_REFERENCE=<checkout> python baseline/make_train_cfg.py"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", "tests", "golden"))
import ref_harness as H  # noqa: E402  (fake isaacgym + reference import paths)

_, _, CfgPPO = H.import_reference_env()
from legged_gym.utils.helpers import class_to_dict  # noqa: E402

train = class_to_dict(CfgPPO())
out = dict(policy=train["policy"], algorithm=train["algorithm"], runner={k: train["runner"][k] for k in ("num_steps_per_env", "policy_class_name", "algorithm_class_name")},
           actor_critic_args=dict(num_actor_obs=76, num_critic_obs=76, num_actions=18, num_priv=24, num_hist=10, num_prop=76),
           source="legged_gym/envs/widowGo1/widowGo1_config.py WidowGo1RoughCfgPPO via legged_gym.utils.helpers.class_to_dict")
json.dump(out, open(os.path.join(HERE, "widowgo1_train_cfg.json"), "w"), indent=1, sort_keys=True)
print(json.dumps(out, indent=1, sort_keys=True))
