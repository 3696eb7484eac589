"""Generate tests/golden/*.npz by running the LIVE Python reference with injected draws.

Needs a checkout of the original project:
    INVERSUS_REFERENCE_ROOT=<checkout> python tests/golden/make_golden.py
The fixtures are the reference's own outputs; oracle/ and the CUDA path are both checked
against them (tests/test_oracle_golden.py, tests/test_cuda_parity.py).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from ref_harness import ReferenceRunner, reference_available  # noqa: E402
from scenarios import SCENARIOS, run_scenario  # noqa: E402


class ReferenceBackend:
    def __init__(self, sc):
        self.r = ReferenceRunner(sc["n"], sc["mode"], sc["difficulty"], sc["max_steps"], seed=sc["seed"])
        self.selfplay = sc["mode"] == "selfplay"

    def reset(self, table):
        self.r.reset(table)

    def step(self, a1, a2, table, auto_reset):
        return self.r.step(a1, a2, table, auto_reset)

    def reset_envs(self, idx, table):
        for i in idx:
            self.r.reset_env(int(i), None if table is None else table[int(i)])

    def state(self):
        return self.r.state()

    def obs(self):
        from inversus.game_types import PlayerId
        ew = self.r.ew
        o1 = [ew.build_observation(e.env, PlayerId.P1) for e in self.r.envs]
        o2 = [ew.build_observation(e.env, PlayerId.P2) for e in self.r.envs]
        return (np.stack([o[0] for o in o1]), np.stack([o[1] for o in o1]),
                np.stack([o[0] for o in o2]), np.stack([o[1] for o in o2]))


def main():
    assert reference_available(), "set INVERSUS_REFERENCE_ROOT to a checkout of the original project"
    only = sys.argv[1:]
    for name, sc in SCENARIOS.items():
        if only and name not in only:
            continue
        be = ReferenceBackend(sc)
        rec = run_scenario(be, sc)
        be.r.close()
        path = os.path.join(HERE, f"{name}.npz")
        np.savez_compressed(path, **rec)
        ndone = int(rec["done"].sum())
        print(f"{name}: {sc['n']} envs x {sc['T']} steps, {ndone} episode ends, "
              f"max bullets {int(rec['state']['n_bullets'].max())}, {os.path.getsize(path)/1024:.0f} KiB")


if __name__ == "__main__":
    main()
