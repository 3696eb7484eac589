"""Golden vectors for GAE from the LIVE reference PPOAgent.compute_advantages
(inversus_rl/ppo_agent.py:127-157). Needs a checkout of the original project:
    INVERSUS_REFERENCE_ROOT=<checkout> python tests/golden/make_gae_golden.py
Writes tests/golden/gae_reference.npz."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from ref_harness import import_reference  # noqa: E402

import_reference()
from inversus_rl.ppo_agent import PPOAgent  # noqa: E402
import torch.nn as nn  # noqa: E402


def main():
    rs = np.random.RandomState(42)
    out = {}
    for case, (m, p_done) in {"a": (2048, 0.02), "b": (777, 0.2), "c": (64, 0.0)}.items():
        agent = PPOAgent(nn.Linear(1, 1))
        r = (rs.randn(m) * 0.5).astype(np.float32)
        v = rs.randn(m).astype(np.float32)
        d = rs.rand(m) < p_done
        agent.reward_buffer = [float(x) for x in r]
        agent.value_buffer = [float(x) for x in v]
        agent.done_buffer = [bool(x) for x in d]
        adv, ret = agent.compute_advantages()
        out.update({f"{case}_reward": r, f"{case}_value": v, f"{case}_done": d.astype(np.uint8),
                    f"{case}_adv": adv, f"{case}_ret": ret})
    np.savez_compressed(os.path.join(HERE, "gae_reference.npz"), **out)
    print("wrote gae_reference.npz", {k: v.shape for k, v in out.items() if k.endswith("adv")})


if __name__ == "__main__":
    main()
