"""Cost of the scripted player as a handle-free kernel and of what is built on it, on one GPU.

  1. inv_scripted_actions: time per call by CUDA events (200 launches captured in a CUDA graph,
     replayed 5 times after warm-up) at each env count and seat, with the bytes it moves per env
     (planes 0-2 of the packed state in, 48 B, and one int8 id out) and the bandwidth that implies.
     The packed planes of 1 M envs (48 MB read) fit the 126 MB L2, so repeated calls read them
     from L2, not HBM.
  2. PPO rollout env-steps/s and samples/s at 65 536 envs, 4 epochs, for selfplay, two mixes and
     vs_dummy hard (steady state: the iterations after the first).
  3. Evaluator episodes/s against the hard dummy with seats="p1" and seats="both".

One JSON line per measurement; the first names the card and its power limit (read in the same run).

    python profiles/measure_mix.py [--out profiles/mix_b200.jsonl]
"""
import argparse
import json
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from measure_eval import card  # noqa: E402

BYTES_IN, BYTES_OUT = 48, 1  # load_board reads planes 0-2 (3 x 16 B); one int8 action id


def scripted_kernel(n, seat, iters=200, warmup=20):
    import numpy as np
    import torch
    from inversus_b200 import BatchedInversus
    from inversus_b200.evaluate import scripted_actions
    from inversus_b200.fused_ops import PackedStates
    sim = BatchedInversus(n, "selfplay", "hard", 500, seed=1, device=0, obs_dtype="none", auto_reset=True)
    sim.reset()
    rs = np.random.RandomState(0)
    for _ in range(8):  # spread the envs' counters and positions
        sim.step(torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda(),
                 torch.from_numpy(rs.randint(0, 13, n).astype(np.int8)).cuda())
    view = PackedStates(sim.packed_state, seat)
    out = torch.empty(n, dtype=torch.int8, device="cuda")
    for _ in range(warmup):
        scripted_actions(view, seat=seat, difficulty="hard", seed=1, out=out)
    torch.cuda.synchronize()
    # the launches are captured in a CUDA graph, so the timing is the device's, not the Python call's
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(iters):
            scripted_actions(view, seat=seat, difficulty="hard", seed=1, out=out)
    graph.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (5 * iters)
    del graph
    sim.close()
    b = n * (BYTES_IN + BYTES_OUT)
    return {"what": "inv_scripted_actions", "num_envs": n, "seat": seat, "us_per_call": us,
            "bytes_per_env": BYTES_IN + BYTES_OUT, "bytes_per_call": b, "GB_per_s": b / (us * 1e-6) / 1e9,
            "l2_resident": b <= 126 * 2 ** 20}


def rollout(name, n, iterations, **kw):
    from inversus_b200.training import train
    with tempfile.TemporaryDirectory() as d:
        out = train(num_envs=n, total_steps=n * 128 * iterations, log_dir=d, rollout_steps=128, epochs=4, seed=3,
                    save=False, quiet=True, **kw)
    s = out["steady_state"]
    return {"what": "rollout", "config": name, "num_envs": n, "epochs": 4, "iterations": s["iterations"],
            "rollout_env_steps_per_s": s["rollout_env_steps_per_s"], "samples_per_s": s["samples_per_s"],
            "cuda_graph": out["cuda_graph"]}


def evaluator(n, seats, episodes=4):
    import torch
    from inversus_b200 import InversusCNNPolicy
    from inversus_b200.evaluate import evaluate
    torch.manual_seed(0)
    policy = InversusCNNPolicy().cuda().eval()
    res = evaluate(policy, "hard", n, episodes, seed=0, seats=seats)
    return {"what": "evaluate", "opponent": "hard", "seats": seats, "num_envs": n, "episodes_per_env": episodes,
            **{k: res[k] for k in ("episodes", "wall_s", "episodes_per_s", "env_steps_per_s")}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[65536, 1048576], help="env counts of the kernel timing")
    ap.add_argument("--num_envs", type=int, default=65536, help="env count of the rollout and evaluator runs")
    ap.add_argument("--iterations", type=int, default=3, help="PPO iterations per rollout configuration")
    ap.add_argument("--kernel-only", action="store_true", help="only the inv_scripted_actions timing")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("measure_mix: needs a CUDA device")
    lines = []

    def emit(row):
        lines.append(row)
        print(json.dumps(row), flush=True)

    emit({"card": card()})
    for n in a.sizes:
        for seat in (0, 1):
            emit(scripted_kernel(n, seat))
    if a.kernel_only:
        return _write(a.out, lines)
    n = a.num_envs
    emit(rollout("selfplay", n, a.iterations, mode="selfplay"))
    emit(rollout("hard=0.5,latest=0.5", n, a.iterations, mode="selfplay", opponent_mix="hard=0.5,latest=0.5"))
    emit(rollout("hard=0.25,latest=0.25,pool=0.5 (pool_size 4)", n, a.iterations, mode="selfplay",
                 opponent_mix="hard=0.25,latest=0.25,pool=0.5", pool_size=4))
    emit(rollout("vs_dummy hard", n, a.iterations, mode="vs_dummy", opponent_difficulty="hard"))
    for seats in ("p1", "both"):
        emit(evaluator(n, seats))
    _write(a.out, lines)


def _write(path, lines):
    if path:
        with open(path, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
