"""Throughput of the evaluator (inversus_b200.evaluate) on one GPU.

For each env count and opponent: one full `evaluate` run (random-init InversusCNNPolicy, K episodes
per env, greedy) for episodes/s and env-steps/s, then a separate eager loop of the same four phases
timed with CUDA events to give each phase's share of the step time. One JSON line per
configuration, the first line names the card and its power limit (read in the same run).

    python profiles/measure_eval.py --sizes 65536 1048576 --episodes 4 [--out profiles/eval.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        smi = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        smi = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(), "nvidia_smi_name_power_limit_max_sm_clock": smi}


def phase_shares(policy, opponent, n, seed, steps=48, warmup=8):
    """Per-phase GPU time of the eager evaluator step (inference, select, step, tally)."""
    import torch
    from inversus_b200 import BatchedInversus
    from inversus_b200.evaluate import episode_tally, select_actions
    from inversus_b200.fused_ops import PackedStates
    h2h = opponent == "policy"
    sim = BatchedInversus(n, "selfplay" if h2h else "dummy", "easy" if h2h else opponent, 500, seed=seed, device=0,
                          obs_dtype="none", auto_reset=True)
    sim.reset()
    views = (PackedStates(sim.packed_state, 0), PackedStates(sim.packed_state, 1))
    counts = torch.zeros((4, n), dtype=torch.int32, device="cuda")
    ret = torch.zeros(n, dtype=torch.float64, device="cuda")
    rem = torch.zeros(1, dtype=torch.int32, device="cuda")
    logits = [torch.empty((n, 13), device="cuda") for _ in range(2)]
    ch = 65536
    names = ("inference", "select", "step", "tally")
    total = dict.fromkeys(names, 0.0)
    for it in range(warmup + steps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        ev[0].record()
        with torch.no_grad():
            for v in range(2 if h2h else 1):
                for a in range(0, n, ch):
                    logits[v][a:min(a + ch, n)].copy_(policy.infer(views[v].chunk(a, min(a + ch, n)), None)[0])
        ev[1].record()
        acts = [select_actions(logits[v], views[v], seed=seed, seat=v, greedy=True) for v in range(2 if h2h else 1)]
        ev[2].record()
        sim.step(acts[0], acts[1] if h2h else None)
        ev[3].record()
        episode_tally(sim, 4, counts, ret, rem)
        ev[4].record()
        torch.cuda.synchronize()
        if it >= warmup:
            for k, name in enumerate(names):
                total[name] += ev[k].elapsed_time(ev[k + 1])
    sim.close()
    step_ms = sum(total.values()) / steps
    return {"eager_step_ms": step_ms,
            "share": {k: v / steps / step_ms for k, v in total.items()},
            "ms": {k: v / steps for k, v in total.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[65536, 1048576])
    ap.add_argument("--opponents", nargs="+", default=["hard", "policy"], help="hard / easy / policy (head to head)")
    ap.add_argument("--episodes", type=int, default=4)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("measure_eval: needs a CUDA device")
    from inversus_b200 import InversusCNNPolicy
    from inversus_b200.evaluate import evaluate
    torch.manual_seed(a.seed)
    policy = InversusCNNPolicy().cuda().eval()
    lines = [{"card": card()}]
    print(json.dumps(lines[0]), flush=True)
    for n in a.sizes:
        for opp in a.opponents:
            res = evaluate(policy, policy if opp == "policy" else opp, n, a.episodes, actions="greedy", seed=a.seed)
            row = {"num_envs": n, "opponent": opp, "episodes_per_env": a.episodes,
                   **{k: res[k] for k in ("episodes", "wins", "losses", "draws", "score", "mean_episode_length",
                                          "env_steps", "wall_s", "env_steps_per_s", "episodes_per_s")},
                   "cuda_graph": n <= 8192, "phases": phase_shares(policy, opp, n, a.seed)}
            lines.append(row)
            print(json.dumps(row), flush=True)
    if a.out:
        with open(a.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
