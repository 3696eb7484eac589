"""GPU-resident PPO training loop: trainer glue around the batched simulator (SURVEY.md section 8f).

Mirrors the reference's entry points and flags (inversus_rl/training.py:53 train_vs_dummy, :204
train_selfplay, :378 main; same `--mode/--num_envs/--total_steps/--log_dir/--opponent_difficulty/
--load_model`, same 8-column training_log.csv, same policy_final.pt / checkpoint files, opponent
snapshot every 20 000 steps), but nothing in the rollout leaves the GPU: the policy reads the
simulator's observation buffers, samples int8 action ids, and the fused step kernel consumes them
on the same stream. One process per GPU under torchrun: every rank owns a shard of the envs
(no communication in the step path), gradients are averaged with one NCCL all-reduce per
minibatch and the four rollout statistics with one more.

    python -m inversus_b200.training --mode vs_dummy --num_envs 4 --total_steps 100000     # README quickstart
    torchrun --nproc-per-node 8 -m inversus_b200.training --num_envs 8388608 --opponent_difficulty hard ...
    python -m inversus_b200.training --mode selfplay --opponent_mix "hard=0.25,latest=0.25,pool=0.5" --pool_size 4 ...
"""
from __future__ import annotations

import argparse
import csv
import os
import time
from collections import deque
from typing import Optional

import torch

from .constants import INFO_LOSE, INFO_WIN
from .policies import InversusCNNPolicy
from .ppo_agent import DeviceRollout, PPOAgent
from .sharding import (dist_env, finish_distributed, init_distributed, opponent_ranges, reduce_rollout_stats,
                       shard_range, sum_over_ranks)
from .simulator import BatchedInversus

OPPONENT_UPDATE_FREQ = 20000  # training.py:265


class TrainingLogger:
    """training.py:16-50: the same training_log.csv columns, so visualize_training.py keeps working;
    throughput goes to a second file."""

    COLUMNS = ["step", "episode", "avg_reward", "win_rate", "avg_ep_len", "policy_loss", "value_loss", "entropy"]

    def __init__(self, log_dir: str):
        os.makedirs(log_dir, exist_ok=True)
        self.log_dir = log_dir
        self.csv_path = os.path.join(log_dir, "training_log.csv")
        self.perf_path = os.path.join(log_dir, "throughput_log.csv")
        with open(self.csv_path, "w", newline="") as f:
            csv.writer(f).writerow(self.COLUMNS)
        with open(self.perf_path, "w", newline="") as f:
            csv.writer(f).writerow(["step", "elapsed_s", "samples_per_s", "rollout_env_steps_per_s", "update_s"])

    def log(self, step, episode, avg_reward, win_rate, avg_ep_len, policy_loss=0.0, value_loss=0.0, entropy=0.0):
        with open(self.csv_path, "a", newline="") as f:
            csv.writer(f).writerow([step, episode, avg_reward, win_rate, avg_ep_len, policy_loss, value_loss, entropy])

    def log_perf(self, step, elapsed, samples_per_s, rollout_rate, update_s):
        with open(self.perf_path, "a", newline="") as f:
            csv.writer(f).writerow([step, elapsed, samples_per_s, rollout_rate, update_s])


class OpponentLogger:
    """opponent_log.csv of a mixed-opponent run: one row per opponent and logging window."""

    COLUMNS = ["step", "opponent", "episodes", "wins", "losses", "draws", "win_rate", "avg_ep_len"]

    def __init__(self, log_dir: str):
        self.path = os.path.join(log_dir, "opponent_log.csv")
        with open(self.path, "w", newline="") as f:
            csv.writer(f).writerow(self.COLUMNS)

    def log(self, step, rows):
        with open(self.path, "a", newline="") as f:
            w = csv.writer(f)
            for name, r in rows.items():
                w.writerow([step, name, r["episodes"], r["wins"], r["losses"], r["draws"], r["win_rate"], r["avg_ep_len"]])


def _opponent_rates(wins: int, losses: int, draws: int, length_sum: int) -> dict:
    n = wins + losses + draws
    return {"episodes": n, "wins": wins, "losses": losses, "draws": draws,
            "win_rate": wins / n if n else 0.0, "avg_ep_len": length_sum / n if n else 0.0}


def train(mode: str = "vs_dummy", num_envs: int = 1, total_steps: int = 500_000, log_dir: Optional[str] = None,
          opponent_difficulty: str = "easy", load_model: Optional[str] = None, *, precision: str = "bf16",
          rollout_steps: Optional[int] = None, batch_size: Optional[int] = None, epochs: int = 4, lr: float = 1e-4,
          reference_gae: bool = False, seed: Optional[int] = None, max_episode_steps: int = 500,
          save: bool = True, quiet: bool = False, cuda_graph: Optional[bool] = None,
          graph_update: bool = True, packed_encoder: Optional[bool] = None, time_allreduce: bool = False,
          opponent_mix=None, pool_size: int = 4) -> dict:
    """Shared body of train_vs_dummy / train_selfplay. `num_envs` is the GLOBAL env count; under
    torchrun each rank simulates its shard. Returns a summary dict (steps, episodes, win_rate,
    samples_per_s, ...).

    opponent_mix (selfplay, bf16 packed-encoder path only), e.g. "hard=0.25,latest=0.25,pool=0.5":
    every env faces one fixed opponent chosen by its global id (sharding.opponent_ranges): the
    scripted dummy ("easy", "hard", through inv_scripted_actions), the lagged copy of the learner
    ("latest", refreshed every OPPONENT_UPDATE_FREQ steps) or one of `pool_size` older snapshots
    ("pool"; at each refresh the oldest is replaced). Per-opponent results go to opponent_log.csv
    and summary["per_opponent"]."""
    assert mode in ("vs_dummy", "selfplay")
    ranges = _check_mix(mode, num_envs, opponent_mix, pool_size, precision, packed_encoder)
    rank, local_rank, world = init_distributed()
    dev = torch.device("cuda", local_rank if world > 1 else torch.cuda.current_device())
    first, n_local = shard_range(num_envs, rank, world)
    log_dir = log_dir or f"runs/inversus_{mode}_envs{num_envs}"
    say = (lambda *a: None) if (quiet or rank != 0) else print
    say(f"Training {mode} with num_envs={num_envs} ({world} GPU(s), {n_local} envs on this rank), "
        f"total_steps={total_steps}, log_dir={log_dir}, precision={precision}")

    if seed is not None:
        torch.manual_seed(seed + rank)
    if precision == "fp32":  # the parity path: real fp32 convolutions, not TF32
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
    selfplay = mode == "selfplay" and ranges is None  # the reference's scheme: one lagged copy for every env
    # bf16 runs feed the policy from the 80-byte packed states (csrc/encoder_kernels.cu): the
    # simulator then keeps no observation tensor at all and a step moves ~200 bytes per env
    if packed_encoder is None:
        packed_encoder = precision == "bf16"
    packed_encoder = bool(packed_encoder) and precision == "bf16"
    sim = BatchedInversus(n_local, "dummy" if mode == "vs_dummy" else "selfplay", opponent_difficulty, max_episode_steps,
                          seed=seed, device=dev.index,
                          obs_dtype="none" if packed_encoder else ("bf16" if precision == "bf16" else "f32"),
                          auto_reset=True, env_id_base=first)
    policy = InversusCNNPolicy()
    if load_model:  # training.py:83-90
        policy.load_state_dict(torch.load(load_model, map_location="cpu"))
        say(f"Loaded {load_model}")
    if world > 1:  # identical initial weights on every rank
        policy = policy.to(dev)
        for p in policy.parameters():
            torch.distributed.broadcast(p.data, src=0)
    target_policy = None
    if selfplay:  # training.py:237-240: the opponent starts as a clone of the learner
        target_policy = InversusCNNPolicy().to(dev)
        target_policy.load_state_dict(policy.state_dict())
        target_policy.eval()
    # mixed opponents: this rank's part of every global range; a policy is built only for the
    # slots that have one, so a purely scripted mix draws from torch's generator exactly as vs_dummy
    segments, pool, pool_oldest = [], [], 0
    if ranges is not None:
        pool = [_clone_policy(policy, dev) for _ in range(pool_size)] if any(
            name.startswith("pool") for name, _, _ in ranges) else []
        if any(name == "latest" for name, _, _ in ranges):
            target_policy = _clone_policy(policy, dev)
        for name, lo, hi in ranges:
            a, b = max(lo, first) - first, min(hi, first + n_local) - first
            net = target_policy if name == "latest" else pool[int(name[5:-1])] if name.startswith("pool") else None
            player = name if net is None else (lambda ps, net=net: net.infer(ps, None)[0])
            segments.append((name, player, max(a, 0), max(b, 0)))

    # training.py:105-107: at least 2048 samples and 128 steps per env per update
    steps_per_env = rollout_steps or max(2048 // max(num_envs, 1), 128)
    if batch_size is None:
        batch_size = 512 if num_envs * steps_per_env <= 1 << 16 else 16384
    agent = PPOAgent(policy, lr=lr, epochs=epochs, batch_size=batch_size, device=str(dev), precision=precision,
                     gae_mode="reference" if reference_gae else "per_env", graph_update=graph_update,
                     packed_encoder=packed_encoder)
    rollout = DeviceRollout(steps_per_env, n_local, dev, store="packed")
    logger = TrainingLogger(log_dir) if rank == 0 else None

    if packed_encoder:
        from .fused_ops import PackedStates
        view_p1, view_p2 = PackedStates(sim.packed_state, 0), PackedStates(sim.packed_state, 1)
    if ranges is not None:
        from .evaluate import seat_actions
        a2_buf = torch.empty(n_local, dtype=torch.int8, device=dev)
        logits2 = torch.empty((n_local, 13), dtype=torch.float32, device=dev) if (target_policy is not None or pool) else None
        # per env since the last log: wins, losses, draws, length sum of P1's finished episodes
        opp_counts = torch.zeros((4, n_local), dtype=torch.int32, device=dev)
        opp_total = {name: [0, 0, 0, 0] for name, _, _ in ranges}
        opp_logger = OpponentLogger(log_dir) if rank == 0 else None

    def observe():
        """What the policy acts on: the live packed state (encoder path) or the observation buffers."""
        return (view_p1, None) if packed_encoder else (sim.obs, sim.extra)

    sim.reset()
    obs, extra = observe()
    step_count = last_log_step = last_opponent_update = episode_count = 0
    recent = deque(maxlen=100)  # (return, length, win) of the last 100 episodes (training.py:164-166)
    exact_recent = num_envs <= 256 and world == 1
    acc = torch.zeros(4, dtype=torch.float64, device=dev)  # episodes, wins, return sum, length sum (since last log)
    update_stats: dict = {}
    window = {"steps": 0, "episodes": 0.0, "wins": 0.0}  # last logging window (all ranks)
    window_start_step = 0
    t_start = time.time()
    rollout_time = update_time = 0.0
    rollout_env_steps = 0
    iters = []      # (samples, rollout seconds, update seconds) per iteration
    iter_steps = 0

    # Small batches are launch-bound (~60 kernels per env step: policy inference, sampling, the
    # fused step, rollout stores). There the whole step is captured ONCE in a CUDA graph and
    # replayed; the time index of the rollout lives on the device so the graph is step-invariant.
    if cuda_graph is None:
        cuda_graph = n_local <= 8192
    exact_recent = exact_recent and not cuda_graph
    t_dev = torch.zeros(1, dtype=torch.int64, device=dev)
    step_graph = None

    def opponent_actions():
        # P2's view of the pre-step state (env_wrappers.py:311) is what the last step/reset emitted
        with torch.no_grad():
            fwd = target_policy.infer if precision == "bf16" else target_policy
            ch = agent.act_chunk
            if packed_encoder:
                parts = [fwd(view_p2.chunk(i, min(i + ch, n_local)), None)[0] for i in range(0, n_local, ch)]
            else:
                parts = [fwd(sim.obs_p2[i:i + ch], sim.extra_p2[i:i + ch])[0] for i in range(0, n_local, ch)]
            logits = parts[0] if len(parts) == 1 else torch.cat(parts)
            # Categorical(logits).sample() without its argument validation (a host sync that a CUDA
            # graph cannot capture); training.py:255-257
            return torch.multinomial(torch.softmax(logits, dim=-1), 1).squeeze(1).to(torch.int8)

    def mixed_opponent_actions():
        # P2's ids slot by slot: the scripted dummy, or a policy's logits sampled by inv_select_actions
        return seat_actions(view_p2, [(player, lo, hi) for _, player, lo, hi in segments], seat=1, seed=sim.seed,
                            gid_base=first, out=a2_buf, logits=logits2, greedy=False, act_chunk=agent.act_chunk)

    def p2_actions():
        return mixed_opponent_actions() if ranges is not None else opponent_actions() if selfplay else None

    def count_opponent_results(d):
        # element-wise per env; reduced per opponent only at the logging point
        win, lose = (sim.info & INFO_WIN) != 0, (sim.info & INFO_LOSE) != 0
        opp_counts[:3].add_(torch.stack([win, lose, d & ~win & ~lose]).to(torch.int32))
        opp_counts[3].add_(torch.where(d, sim.episode_steps, 0))

    def graphed_step():
        actions, log_probs, values = agent.act(obs, extra)
        rollout.store_pre_at(t_dev, sim, actions, log_probs, values)
        a2 = p2_actions()
        sim.step(actions.to(torch.int8), a2)
        rollout.store_post_at(t_dev, sim.reward, sim.done)
        d = sim.done.bool()
        acc.add_(torch.stack([d.sum(), ((sim.info & INFO_WIN) != 0).sum(),
                              torch.where(d, sim.episode_return, 0.0).sum(),
                              torch.where(d, sim.episode_steps, 0).sum()]).to(torch.float64))
        if ranges is not None:
            count_opponent_results(d)
        t_dev.add_(1)

    if cuda_graph:
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(3):
                t_dev.zero_()
                graphed_step()
        torch.cuda.current_stream(dev).wait_stream(side)
        step_graph = torch.cuda.CUDAGraph()
        t_dev.zero_()
        with torch.cuda.graph(step_graph):
            graphed_step()
        sim.reset()  # warm-up and capture stepped the envs: start fresh episodes
        obs, extra = observe()
        acc.zero_()
        if ranges is not None:
            opp_counts.zero_()

    while step_count < total_steps:
        t0 = time.time()
        if cuda_graph:
            t_dev.zero_()
            n_steps = min(steps_per_env, -(-(total_steps - step_count) // num_envs))
            for _ in range(n_steps):
                step_graph.replay()
            rollout.t = n_steps
            step_count += n_steps * num_envs
            rollout_env_steps += n_steps * num_envs
        for _ in range(0 if cuda_graph else steps_per_env):
            actions, log_probs, values = agent.act(obs, extra)
            rollout.store_pre(sim, actions, log_probs, values)
            a2 = p2_actions()
            _, rewards, dones, info = sim.step(actions.to(torch.int8), a2)
            obs, extra = observe()
            rollout.store_post(rewards, dones)
            d = dones.bool()
            acc += torch.stack([d.sum(), ((info & INFO_WIN) != 0).sum(),
                                torch.where(d, sim.episode_return, 0.0).sum(),
                                torch.where(d, sim.episode_steps, 0).sum()]).to(torch.float64)
            if ranges is not None:
                count_opponent_results(d)
            if exact_recent:  # small runs: the reference's exact last-100-episodes window
                dn = d.nonzero().flatten().tolist()
                if dn:
                    er, es, inf = sim.episode_return.tolist(), sim.episode_steps.tolist(), info.tolist()
                    for i in dn:
                        recent.append((er[i], es[i], 1 if inf[i] & INFO_WIN else 0))
            step_count += num_envs
            rollout_env_steps += num_envs
            if step_count >= total_steps:
                break
        torch.cuda.synchronize(dev)
        t1 = time.time()
        # bootstrap with the value of the state after the last step (per-env GAE only; the
        # reference bootstraps with 0, ppo_agent.py:170)
        last_value = None
        if not reference_gae:
            last_value = agent.act(obs, extra)[2]
        update_stats = agent.update(rollout, sim, last_value)
        if precision == "bf16":
            policy.inference_weights()  # refresh the cached bf16 copies in place (the step graph reads them)
        torch.cuda.synchronize(dev)
        t2 = time.time()
        rollout_time += t1 - t0
        update_time += t2 - t1
        iters.append((rollout.T * num_envs if not iters else step_count - iter_steps, t1 - t0, t2 - t1))
        iter_steps = step_count

        if selfplay and step_count - last_opponent_update >= OPPONENT_UPDATE_FREQ:  # training.py:331-334
            target_policy.load_state_dict(policy.state_dict())
            if precision == "bf16":
                target_policy.inference_weights()
            last_opponent_update = step_count
        if ranges is not None and step_count - last_opponent_update >= OPPONENT_UPDATE_FREQ:
            # in place (same bf16 tensors), so a captured step graph keeps working
            for net in ([target_policy] if target_policy is not None else []) + pool[pool_oldest:pool_oldest + 1]:
                net.load_state_dict(policy.state_dict())
                net.inference_weights()
            if pool:
                pool_oldest = (pool_oldest + 1) % len(pool)
            last_opponent_update = step_count

        if step_count - last_log_step >= 1000 or step_count >= total_steps:  # training.py:172
            ep, wins, rsum, lsum = reduce_rollout_stats(*acc.tolist(), device=dev)
            acc.zero_()
            if ranges is not None:
                per_slot = torch.stack([opp_counts[:, lo:hi].sum(1) for _, _, lo, hi in segments]).to(torch.int64)
                opp_counts.zero_()
                window_rows = {}
                for (name, _, _, _), row in zip(segments, sum_over_ranks(per_slot).tolist()):
                    opp_total[name] = [t + v for t, v in zip(opp_total[name], row)]
                    window_rows[name] = _opponent_rates(*row)
            episode_count += int(ep)
            window = {"steps": step_count - window_start_step, "episodes": ep, "wins": wins}
            window_start_step = step_count
            if exact_recent and recent:
                avg_reward = sum(r for r, _, _ in recent) / len(recent)
                avg_len = sum(s for _, s, _ in recent) / len(recent)
                win_rate = sum(w for _, _, w in recent) / len(recent)
            else:
                avg_reward, avg_len, win_rate = (rsum / ep, lsum / ep, wins / ep) if ep > 0 else (0.0, 0.0, 0.0)
            elapsed = time.time() - t_start
            last_log_step = step_count  # on EVERY rank: the branch above contains a collective
            if rank == 0 and episode_count > 0:
                logger.log(step_count, episode_count, avg_reward, win_rate, avg_len, update_stats.get("policy_loss", 0.0),
                           update_stats.get("value_loss", 0.0), update_stats.get("entropy", 0.0))
                logger.log_perf(step_count, elapsed, step_count / elapsed, rollout_env_steps / max(rollout_time, 1e-9),
                                t2 - t1)
                if ranges is not None:
                    opp_logger.log(step_count, window_rows)
                say(f"Step {step_count}/{total_steps} | Episodes: {episode_count} | Avg Reward: {avg_reward:.3f} | "
                    f"Win Rate: {win_rate:.3f} | Avg Ep Len: {avg_len:.1f} | Time: {elapsed:.1f}s | "
                    f"{step_count / elapsed:,.0f} samples/s")
            if save and rank == 0 and step_count % 50000 == 0 and step_count > 0:  # training.py:193
                torch.save(policy.state_dict(), os.path.join(log_dir, f"policy_checkpoint_{step_count}.pt"))

    elapsed = time.time() - t_start
    if save and rank == 0:
        torch.save(policy.state_dict(), os.path.join(log_dir, "policy_final.pt"))  # training.py:199-200
    allreduce = agent.time_allreduce() if (time_allreduce and world > 1) else None
    summary = {"steps": step_count, "episodes": episode_count, "elapsed_s": elapsed, "allreduce": allreduce,
               "packed_encoder": packed_encoder, "epochs": epochs,
               "samples_per_s": step_count / elapsed, "rollout_s": rollout_time, "update_s": update_time,
               "rollout_env_steps_per_s": rollout_env_steps / max(rollout_time, 1e-9),
               "win_rate": win_rate if episode_count else None, "avg_reward": avg_reward if episode_count else None,
               "avg_ep_len": avg_len if episode_count else None, **update_stats,
               "steady_state": _steady(iters),
               "last_window": window,
               "wins_per_kstep": 1e3 * window["wins"] / max(window["steps"], 1),
               "n_gpus": world, "num_envs": num_envs, "steps_per_env": steps_per_env, "batch_size": batch_size,
               "precision": precision, "cuda_graph": bool(cuda_graph)}
    if ranges is not None:
        summary["per_opponent"] = {name: _opponent_rates(*t) for name, t in opp_total.items()}
        summary["opponent_ranges"] = ranges
    sim.close()
    return summary


def _check_mix(mode, num_envs, opponent_mix, pool_size, precision, packed_encoder):
    """The global opponent ranges of a mixed-opponent run (None without a mix); ValueError on a bad
    combination."""
    if opponent_mix is None:
        if pool_size != 4:
            raise ValueError("pool_size is only valid with opponent_mix")
        return None
    if mode != "selfplay":
        raise ValueError("opponent_mix is only valid with mode='selfplay'")
    if precision != "bf16" or packed_encoder is False:
        raise ValueError("opponent_mix needs the bf16 packed-encoder path (its opponents read the packed state)")
    return opponent_ranges(num_envs, opponent_mix, pool_size)


def _clone_policy(policy: InversusCNNPolicy, dev) -> InversusCNNPolicy:
    """An opponent that starts as a copy of the learner (training.py:237-240)."""
    net = InversusCNNPolicy().to(dev)
    net.load_state_dict(policy.state_dict())
    return net.eval()


def _steady(iters):
    """Throughput over the iterations after the first (which pays cuDNN/NCCL/allocator warm-up)."""
    body = iters[1:] if len(iters) > 1 else iters
    n, r, u = (sum(x[i] for x in body) for i in range(3))
    return {"iterations": len(body), "samples": n, "rollout_s": r, "update_s": u,
            "samples_per_s": n / max(r + u, 1e-9), "rollout_env_steps_per_s": n / max(r, 1e-9),
            "update_samples_per_s": n / max(u, 1e-9)}


def train_vs_dummy(num_envs: int = 1, total_steps: int = 500_000, log_dir: str = "runs/inversus_vs_dummy",
                   opponent_difficulty: str = "easy", load_model: Optional[str] = None, **kw) -> dict:
    """training.py:53-201."""
    return train("vs_dummy", num_envs, total_steps, log_dir, opponent_difficulty, load_model, **kw)


def train_selfplay(num_envs: int = 1, total_steps: int = 500_000, log_dir: str = "runs/inversus_selfplay",
                   load_model: Optional[str] = None, **kw) -> dict:
    """training.py:204-375."""
    return train("selfplay", num_envs, total_steps, log_dir, "easy", load_model, **kw)


def main(argv=None):
    """training.py:378-407 -- same flags; `--num_envs` is no longer capped at 16."""
    ap = argparse.ArgumentParser(description="Train INVERSUS RL agent (GPU-resident rollout)")
    ap.add_argument("--mode", choices=["vs_dummy", "selfplay"], default="vs_dummy")
    ap.add_argument("--num_envs", type=int, default=1, help="Number of parallel environments (global)")
    ap.add_argument("--total_steps", type=int, default=500000)
    ap.add_argument("--log_dir", type=str, default=None)
    ap.add_argument("--opponent_difficulty", type=str, default="easy", choices=["easy", "hard"])
    ap.add_argument("--load_model", type=str, default=None)
    ap.add_argument("--precision", choices=["bf16", "fp32"], default="bf16")
    ap.add_argument("--rollout_steps", type=int, default=None, help="env steps per update (default: reference rule)")
    ap.add_argument("--batch_size", type=int, default=None)
    ap.add_argument("--reference-gae", action="store_true", help="flat-list GAE exactly like ppo_agent.py:127-157")
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--cuda-graph", choices=["auto", "on", "off"], default="auto",
                    help="capture one rollout step in a CUDA graph (auto: when <= 8192 envs per GPU)")
    ap.add_argument("--opponent_mix", type=str, default=None,
                    help='selfplay only: per-env opponents by global id, e.g. "hard=0.25,latest=0.25,pool=0.5" '
                         "(slots easy, hard, latest, pool)")
    ap.add_argument("--pool_size", type=int, default=None, help="snapshots in the pool slot of --opponent_mix (4)")
    a = ap.parse_args(argv)
    if a.pool_size is not None and a.opponent_mix is None:
        ap.error("--pool_size is only valid with --opponent_mix")
    try:
        _check_mix(a.mode, a.num_envs, a.opponent_mix, 4 if a.pool_size is None else a.pool_size, a.precision, None)
    except ValueError as e:
        ap.error(str(e))
    log_dir = a.log_dir or f"runs/inversus_{a.mode}_envs{a.num_envs}"
    out = train(a.mode, a.num_envs, a.total_steps, log_dir, a.opponent_difficulty, a.load_model,
                precision=a.precision, rollout_steps=a.rollout_steps, batch_size=a.batch_size,
                reference_gae=a.reference_gae, seed=a.seed,
                cuda_graph={"auto": None, "on": True, "off": False}[a.cuda_graph], opponent_mix=a.opponent_mix,
                pool_size=4 if a.pool_size is None else a.pool_size)
    if dist_env()[0] == 0:
        print({k: (round(v, 4) if isinstance(v, float) else v) for k, v in out.items()}, flush=True)
    finish_distributed()  # the update graph holds NCCL kernels


if __name__ == "__main__":
    main()
