"""GPU-resident evaluation: play a policy for exactly K episodes per env against the scripted dummy
or against a second policy, and report win rate, score and Elo with 95 % intervals.

The simulator runs with auto-reset and no observation tensor; the policy reads the packed states
(the bf16 path the trainer uses). Per step: inference -> `inv_select_actions` (greedy, or one
counter-based draw per env) -> the fused step -> `inv_episode_tally`, which counts only the first
K episodes of every env, so short episodes are not over-represented. The host reads one integer
every 32 steps; nothing else leaves the GPU until the end (DESIGN.md "evaluator").

    python -m inversus_b200.evaluate --model A.pt --opponent hard --num_envs 65536 --episodes_per_env 4
    python -m inversus_b200.evaluate --model A.pt --opponent hard --seats both ...   # the dummy in either seat
    torchrun --nproc-per-node 8 -m inversus_b200.evaluate --model A.pt --opponent B.pt --num_envs 1048576 ...
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time
from statistics import NormalDist
from typing import Callable, Optional, Tuple

import torch

from . import _capi
from .constants import NUM_ACTIONS, STATUS_INVALID_ACTION
from .fused_ops import PackedStates, _packed_args
from .sharding import finish_distributed, init_distributed, shard_range
from .simulator import BatchedInversus

SCRIPTED = ("easy", "hard")
ACTIONS = ("greedy", "sample")
SEATS = ("p1", "both")
CHECK_EVERY = 32  # steps between the host's reads of the `remaining` counter
Z95 = NormalDist().inv_cdf(0.975)


# ---------------------------------------------------------------------------------------- statistics
def wilson_interval(k: float, n: int, z: float = Z95) -> Tuple[float, float]:
    """Wilson score interval of a proportion k / n (Newcombe 1998; the formula and the end-point
    rule of scipy.stats.binomtest(...).proportion_ci(method="wilson")). k may be fractional."""
    if n <= 0:
        return (float("nan"), float("nan"))
    p = k / n
    denom = 2 * (n + z ** 2)
    center = (2 * n * p + z ** 2) / denom
    delta = z / denom * math.sqrt(4 * n * p * (1 - p) + z ** 2)
    return (0.0 if k == 0 else center - delta, 1.0 if k == n else center + delta)


def score(wins: int, draws: int, n: int) -> float:
    """(wins + draws / 2) / n: the expected points of one game."""
    return (wins + 0.5 * draws) / n


def elo_from_score(s: float) -> Optional[float]:
    """Rating difference that predicts score s under the logistic Elo model; None at s = 0 or 1."""
    if not 0.0 < s < 1.0:
        return None
    return 400.0 * math.log10(s / (1.0 - s))


def _rates(wins: int, losses: int, draws: int, length_sum: int) -> dict:
    n = wins + losses + draws
    out = {"episodes": n, "wins": wins, "losses": losses, "draws": draws}
    if n == 0:
        return {**out, "win_rate": None, "win_rate_ci95": None, "score": None, "score_ci95": None, "elo": None,
                "elo_ci95": None, "mean_episode_length": None}
    s = score(wins, draws, n)
    s_lo, s_hi = wilson_interval(wins + 0.5 * draws, n)
    return {**out, "win_rate": wins / n, "win_rate_ci95": list(wilson_interval(wins, n)), "score": s,
            "score_ci95": [s_lo, s_hi], "elo": elo_from_score(s), "elo_ci95": [elo_from_score(s_lo), elo_from_score(s_hi)],
            "mean_episode_length": length_sum / n}


# ---------------------------------------------------------------------------------------- kernels
def _stream(device: torch.device) -> int:
    return int(torch.cuda.current_stream(device).cuda_stream)


def select_actions(logits: torch.Tensor, ps: PackedStates, *, seed: int, seat: int = 0, greedy: bool = True,
                   gid_base: int = 0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """int8 action ids from fp32 logits [n, 13] (inv_select_actions). `ps` holds the envs' packed
    states (entry i = env gid_base + i); sampling reads their (episode, step_count) counter words."""
    assert logits.is_cuda and logits.dtype == torch.float32 and logits.dim() == 2 and logits.shape[1] == NUM_ACTIONS
    assert logits.is_contiguous() and logits.shape[0] == len(ps)
    n = logits.shape[0]
    if out is None:
        out = torch.empty(n, dtype=torch.int8, device=logits.device)
    assert out.dtype == torch.int8 and out.is_contiguous() and out.numel() == n
    ptr, stride, count = _packed_args(ps)
    with torch.cuda.device(logits.device):
        _capi.check(_capi.load().inv_select_actions(logits.data_ptr(), count, ptr, stride, int(gid_base),
                                                    int(seed) & 0xFFFFFFFFFFFFFFFF, int(seat), int(bool(greedy)),
                                                    out.data_ptr(), _stream(logits.device)))
    return out


def scripted_actions(ps: PackedStates, *, seat: int, difficulty, seed: int, gid_base: int = 0,
                     out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """int8 action ids of the scripted dummy playing `seat` (0 = P1, 1 = P2) on the envs of `ps`
    (entry i = env gid_base + i), from their pre-step packed states (inv_scripted_actions). Seat 1
    is exactly the opponent of a dummy-mode step. difficulty: "easy" / "hard" (or 0 / 1)."""
    difficulty = _capi.DIFFICULTY[difficulty] if isinstance(difficulty, str) else int(difficulty)
    dev = ps.planes.device
    n = len(ps)
    if out is None:
        out = torch.empty(n, dtype=torch.int8, device=dev)
    assert out.dtype == torch.int8 and out.is_contiguous() and out.numel() == n
    ptr, stride, count = _packed_args(ps)
    with torch.cuda.device(dev):
        _capi.check(_capi.load().inv_scripted_actions(ptr, stride, count, int(gid_base), int(seed) & 0xFFFFFFFFFFFFFFFF,
                                                      int(seat), difficulty, out.data_ptr(), _stream(dev)))
    return out


def seat_actions(view: PackedStates, segments, *, seat: int, seed: int, gid_base: int, out: torch.Tensor,
                 logits: Optional[torch.Tensor] = None, greedy: bool = True, act_chunk: int = 65536) -> torch.Tensor:
    """Seat `seat`'s int8 action ids for all envs of `view` (entry i = env gid_base + i), built
    segment by segment into `out`. `segments` lists (player, lo, hi) over [0, len(view)): a player is
    "easy" / "hard" (the scripted dummy, inv_scripted_actions) or a `PackedStates -> logits`
    callable, run in micro-batches of `act_chunk` into the fp32 `logits` buffer [len(view), 13] and
    turned into ids by inv_select_actions (greedy or sampled)."""
    with torch.no_grad():
        for player, lo, hi in segments:
            if lo >= hi:
                continue
            if isinstance(player, str):
                scripted_actions(view.chunk(lo, hi), seat=seat, difficulty=player, seed=seed, gid_base=gid_base + lo,
                                 out=out[lo:hi])
                continue
            for a in range(lo, hi, act_chunk):
                b = min(a + act_chunk, hi)
                logits[a:b].copy_(player(view.chunk(a, b)))
            select_actions(logits[lo:hi], view.chunk(lo, hi), seed=seed, seat=seat, greedy=greedy,
                           gid_base=gid_base + lo, out=out[lo:hi])
    return out


def episode_tally(sim: BatchedInversus, quota: int, counts: torch.Tensor, return_sum: torch.Tensor,
                  remaining: torch.Tensor) -> None:
    """Add the episodes that ended in `sim`'s last step into the per-env accumulators
    (inv_episode_tally): counts int32 [4, n] (wins, losses, draws, length sum from P1's side),
    return_sum f64 [n], and the number of envs still short of `quota` episodes into remaining (int32 [1])."""
    n = sim.num_envs
    assert counts.dtype == torch.int32 and tuple(counts.shape) == (4, n) and counts.is_contiguous()
    assert return_sum.dtype == torch.float64 and return_sum.numel() == n and remaining.dtype == torch.int32
    with torch.cuda.device(sim.device):
        _capi.check(_capi.load().inv_episode_tally(
            sim.done.data_ptr(), sim.info.data_ptr(), sim.episode_steps.data_ptr(), sim.episode_return.data_ptr(),
            sim.packed_state.data_ptr(), n, n, int(quota), sim.max_episode_steps, counts.data_ptr(),
            return_sum.data_ptr(), remaining.data_ptr(), _stream(sim.device)))


# ---------------------------------------------------------------------------------------- players
def _describe(p) -> str:
    if isinstance(p, (str, os.PathLike)):
        return str(p)
    return getattr(p, "__name__", type(p).__name__)


def _logits_fn(p, device: torch.device) -> Callable[[PackedStates], torch.Tensor]:
    """A policy as `PackedStates -> fp32 logits [n, 13]`: an InversusCNNPolicy (bf16 inference
    path), the path of a reference-compatible state dict, or such a callable itself."""
    from .policies import InversusCNNPolicy
    if isinstance(p, (str, os.PathLike)):
        net = InversusCNNPolicy()
        net.load_state_dict(torch.load(p, map_location="cpu"))
        p = net
    if isinstance(p, InversusCNNPolicy):
        net = p.to(device).eval()
        return lambda ps: net.infer(ps, None)[0]
    if callable(p):
        return p
    raise TypeError(f"not a policy: {p!r}")


def _check_args(opponent, num_envs: int, episodes_per_env: int, actions: str, max_episode_steps: int,
                seats: str = "p1") -> bool:
    """Raises ValueError on a bad combination; returns True when the policy plays both seats (head
    to head, or the scripted dummy with seats="both")."""
    if actions not in ACTIONS:
        raise ValueError(f"actions must be one of {ACTIONS}, got {actions!r}")
    if seats not in SEATS:
        raise ValueError(f"seats must be one of {SEATS}, got {seats!r}")
    if isinstance(opponent, str) and opponent not in SCRIPTED and not os.path.isfile(opponent):
        raise ValueError(f"opponent must be 'easy', 'hard', a policy or a checkpoint file, got {opponent!r}")
    head_to_head = not (isinstance(opponent, str) and opponent in SCRIPTED)
    two_seats = head_to_head or seats == "both"
    if episodes_per_env < 1:
        raise ValueError("episodes_per_env must be at least 1")
    if num_envs < (2 if two_seats else 1):
        raise ValueError("head to head needs at least 2 envs (one per seat)" if head_to_head
                         else "seats='both' needs at least 2 envs (one per seat)" if two_seats
                         else "num_envs must be at least 1")
    if max_episode_steps < 1 or episodes_per_env * max_episode_steps >= 1 << 31:
        raise ValueError("episodes_per_env * max_episode_steps must be below 2^31")
    return two_seats


def play_shard(policy, opponent, num_envs: int, episodes_per_env: int, first: int, count: int, *,
               actions: str = "greedy", seed: int, max_episode_steps: int = 500, act_chunk: Optional[int] = None,
               cuda_graph: Optional[bool] = None, device=None, seats: str = "p1") -> dict:
    """Play the envs with global ids [first, first + count) of an evaluation over `num_envs` envs
    (what one rank does) and return their raw tallies from the policy's side:
    `seats` int64 [2, 4] (rows: policy as P1, policy as P2; columns: wins, losses, draws, length
    sum), `p1_return_sum` (P1's summed episode return over the shard's policy-as-P1 envs),
    `env_steps` and `steps`."""
    two_seats = _check_args(opponent, num_envs, episodes_per_env, actions, max_episode_steps, seats)
    head_to_head = not (isinstance(opponent, str) and opponent in SCRIPTED)
    if not (0 <= first and 1 <= count and first + count <= num_envs):
        raise ValueError("the shard must lie inside [0, num_envs)")
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else torch.device(device).index or 0)
    K, n = int(episodes_per_env), int(count)
    ch = int(act_chunk or 65536)
    greedy = actions == "greedy"
    pol = _logits_fn(policy, dev)
    # the scripted dummy of a seats="both" run plays through inv_scripted_actions, not the step
    opp = _logits_fn(opponent, dev) if head_to_head else opponent
    sim = BatchedInversus(n, "selfplay" if two_seats else "dummy", "easy" if two_seats else opponent,
                          max_episode_steps, seed=seed, device=dev.index, obs_dtype="none", auto_reset=True,
                          env_id_base=first)
    # both seats: global ids [0, ceil(N/2)) seat the policy as P1, the rest as P2
    split = min(max(-(-num_envs // 2) - first, 0), n) if two_seats else n
    seats1 = [(pol, 0, split), (opp, split, n)]  # who plays P1 on which local envs
    seats2 = [(opp, 0, split), (pol, split, n)]
    with torch.cuda.device(dev):
        views = (PackedStates(sim.packed_state, 0), PackedStates(sim.packed_state, 1))
        logits = [torch.empty((n, NUM_ACTIONS), dtype=torch.float32, device=dev) for _ in range(2)]
        acts = [torch.empty(n, dtype=torch.int8, device=dev) for _ in range(2)]
        counts = torch.zeros((4, n), dtype=torch.int32, device=dev)
        ret = torch.zeros(n, dtype=torch.float64, device=dev)
        remaining = torch.zeros(1, dtype=torch.int32, device=dev)

        def act(view: int, segments) -> torch.Tensor:
            return seat_actions(views[view], segments, seat=view, seed=sim.seed, gid_base=first, out=acts[view],
                                logits=logits[view], greedy=greedy, act_chunk=ch)

        def one_step():
            a1 = act(0, seats1)
            a2 = act(1, seats2) if two_seats else None
            sim.step(a1, a2)
            episode_tally(sim, K, counts, ret, remaining)

        sim.reset()
        graph = None
        if cuda_graph is None:
            cuda_graph = n <= 8192  # launch-bound below this size, as in training.train
        if cuda_graph:
            start = sim.snapshot()
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(3):
                    one_step()
            torch.cuda.current_stream(dev).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                one_step()
            # warm-up and capture stepped the envs: back to the first episode of every env
            sim.restore(start)
            counts.zero_()
            ret.zero_()

        bound = K * max_episode_steps + 1  # every episode ends within max_episode_steps steps
        steps = 0
        while True:
            for _ in range(min(CHECK_EVERY, bound - steps)):
                graph.replay() if graph is not None else one_step()
            steps += min(CHECK_EVERY, bound - steps)
            if int(remaining.item()) == 0:
                break
            if steps >= bound:
                raise _capi.InversusError(f"{int(remaining.item())} envs still short of {K} episodes after {steps} "
                                          f"steps (max_episode_steps={max_episode_steps})")
        bits = sim.poll_status()
        if bits & STATUS_INVALID_ACTION:
            raise _capi.InversusError("a policy produced logits with NaN or +inf, or only -inf: invalid action id")
        if bits:
            raise _capi.InversusError(f"simulator status bits 0x{bits:x} during the evaluation")
        c = counts.to(torch.int64)
        side1 = c[:, :split].sum(1)                     # policy is P1: P1's wins are its wins
        side2 = c[:, split:].sum(1)[[1, 0, 2, 3]]       # policy is P2: P1's losses are its wins
        out = {"seats": torch.stack([side1, side2]).cpu(), "p1_return_sum": ret[:split].sum(),
               "env_steps": steps * n, "steps": steps}
    del graph
    sim.close()
    return out


def evaluate(policy, opponent, num_envs: int, episodes_per_env: int, *, actions: str = "greedy", seed: int,
             max_episode_steps: int = 500, act_chunk: Optional[int] = None, cuda_graph: Optional[bool] = None,
             seats: str = "p1") -> dict:
    """Play `policy` for exactly `episodes_per_env` episodes in each of `num_envs` envs (global
    count; under torchrun every rank plays its `shard_range`) against `opponent`: "easy" / "hard"
    (the scripted dummy) or a second policy, head to head with seats split by global env id.
    A policy is an InversusCNNPolicy, a checkpoint path, or a callable PackedStates -> fp32 logits
    [n, 13]. actions: "greedy" (argmax) or "sample" (one counter-based draw per env and step).
    seats (scripted opponent only): "p1" seats the policy as P1 in every env; "both" splits the
    seats by global env id as head to head does, the dummy playing the other seat. Returns the
    result dict; wins / losses / draws are from `policy`'s side."""
    _check_args(opponent, num_envs, episodes_per_env, actions, max_episode_steps, seats)
    head_to_head = not (isinstance(opponent, str) and opponent in SCRIPTED)
    rank, local_rank, world = init_distributed()
    dev = torch.device("cuda", local_rank if world > 1 else torch.cuda.current_device())
    first, n_local = shard_range(num_envs, rank, world)
    t0 = time.time()
    raw = play_shard(policy, opponent, num_envs, episodes_per_env, first, n_local, actions=actions, seed=seed,
                     max_episode_steps=max_episode_steps, act_chunk=act_chunk, cuda_graph=cuda_graph, device=dev,
                     seats=seats)
    ints = torch.cat([raw["seats"].flatten(), torch.tensor([raw["env_steps"]])]).to(dev)
    rsum = raw["p1_return_sum"].reshape(1).to(dev)
    if world > 1:
        torch.distributed.all_reduce(ints)
        torch.distributed.all_reduce(rsum)
    ints, rsum = ints.tolist(), float(rsum.item())
    wall = time.time() - t0
    per_seat = [ints[0:4], ints[4:8]]
    env_steps = ints[8]
    tot = [per_seat[0][k] + per_seat[1][k] for k in range(4)]
    res = _rates(*tot)
    assert res["episodes"] == num_envs * episodes_per_env, (res["episodes"], num_envs, episodes_per_env)
    # the shaped reward is P1's: its mean over the policy-as-P1 episodes
    p1_episodes = sum(per_seat[0][:3])
    res["mean_return"] = None if head_to_head else rsum / p1_episodes
    res["per_seat"] = {"p1": _rates(*per_seat[0]), "p2": _rates(*per_seat[1])}
    res.update({"env_steps": env_steps, "wall_s": wall, "env_steps_per_s": env_steps / wall,
                "episodes_per_s": res["episodes"] / wall})
    res["args"] = {"policy": _describe(policy), "opponent": _describe(opponent), "num_envs": num_envs,
                   "episodes_per_env": episodes_per_env, "actions": actions, "seed": seed,
                   "max_episode_steps": max_episode_steps, "act_chunk": act_chunk or 65536,
                   "cuda_graph": cuda_graph, "n_gpus": world, "seats": seats}
    return res


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description="Evaluate an INVERSUS policy checkpoint on the GPU")
    ap.add_argument("--model", required=True, help="checkpoint (.pt state dict) of the policy to evaluate")
    ap.add_argument("--opponent", required=True, help="easy, hard (scripted dummy) or a second checkpoint")
    ap.add_argument("--num_envs", type=int, default=4096, help="parallel environments (global)")
    ap.add_argument("--episodes_per_env", type=int, default=1, help="episodes counted in every env (K)")
    ap.add_argument("--actions", choices=ACTIONS, default="greedy")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--max_episode_steps", type=int, default=500)
    ap.add_argument("--act_chunk", type=int, default=None, help="samples per inference micro-batch (65536)")
    ap.add_argument("--cuda-graph", choices=["auto", "on", "off"], default="auto",
                    help="replay one captured step (auto: when <= 8192 envs per GPU)")
    ap.add_argument("--seats", choices=SEATS, default="p1",
                    help="scripted opponent: the policy plays P1 only, or P1 in the first half of the envs "
                         "and P2 in the rest (a policy opponent always plays both)")
    ap.add_argument("--json", default=None, help="also write the result to this file")
    a = ap.parse_args(argv)
    if not os.path.isfile(a.model):
        ap.error(f"--model {a.model}: no such file")
    try:
        _check_args(a.opponent, a.num_envs, a.episodes_per_env, a.actions, a.max_episode_steps, a.seats)
    except ValueError as e:
        ap.error(str(e))
    if not torch.cuda.is_available():
        print("evaluate: no CUDA device: the evaluator has no CPU fallback", file=sys.stderr)
        return 1
    res = evaluate(a.model, a.opponent, a.num_envs, a.episodes_per_env, actions=a.actions, seed=a.seed,
                   max_episode_steps=a.max_episode_steps, act_chunk=a.act_chunk,
                   cuda_graph={"auto": None, "on": True, "off": False}[a.cuda_graph], seats=a.seats)
    if int(os.environ.get("RANK", 0)) == 0:
        line = json.dumps(res)
        print(line, flush=True)
        if a.json:
            with open(a.json, "w") as f:
                f.write(line + "\n")
    finish_distributed()
    return 0


if __name__ == "__main__":
    sys.exit(main())
