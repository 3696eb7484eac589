"""CPU checks of the evaluator (inversus_b200.evaluate): its interval / score / Elo helpers, the
command line's argument checks, and that its two CUDA entry points refuse to run without a device."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("n", [1, 2, 7, 100, 4096, 1 << 20])
def test_wilson_interval_matches_scipy_at_the_edges(n):
    from scipy.stats import binomtest
    from inversus_b200.evaluate import wilson_interval
    for k in sorted({0, 1, n - 1, n // 2, n}):
        want = binomtest(k, n).proportion_ci(confidence_level=0.95, method="wilson")
        lo, hi = wilson_interval(k, n)
        assert abs(lo - want.low) <= 1e-12 and abs(hi - want.high) <= 1e-12, (k, n, (lo, hi), want)


def test_score_and_elo():
    from scipy.stats import binomtest
    from inversus_b200.evaluate import _rates, elo_from_score, score, wilson_interval
    assert score(3, 2, 10) == 0.4 and score(0, 0, 5) == 0.0 and score(5, 0, 5) == 1.0
    assert elo_from_score(0.5) == 0.0
    assert elo_from_score(0.0) is None and elo_from_score(1.0) is None
    assert abs(elo_from_score(10 / 11) - 400.0) < 1e-9          # 10:1 odds = +400
    assert abs(elo_from_score(0.25) + elo_from_score(0.75)) < 1e-12
    # without draws the score interval is the win-rate interval
    r = _rates(wins=37, losses=63, draws=0, length_sum=4321)
    want = binomtest(37, 100).proportion_ci(method="wilson")
    assert r["episodes"] == 100 and r["score"] == r["win_rate"] == 0.37 and r["mean_episode_length"] == 43.21
    assert abs(r["win_rate_ci95"][0] - want.low) <= 1e-12 and abs(r["win_rate_ci95"][1] - want.high) <= 1e-12
    assert r["score_ci95"] == r["win_rate_ci95"]
    assert r["elo_ci95"] == [elo_from_score(want.low), elo_from_score(want.high)]
    # draws count half; the interval is Wilson's at the fractional count
    r = _rates(wins=10, losses=20, draws=10, length_sum=0)
    assert r["score"] == 15 / 40 and r["score_ci95"] == list(wilson_interval(15.0, 40))
    r = _rates(0, 0, 0, 0)
    assert r["episodes"] == 0 and r["win_rate"] is None and r["score"] is None


def _cli(*args):
    return subprocess.run([sys.executable, "-m", "inversus_b200.evaluate", *args], cwd=ROOT, capture_output=True,
                          text=True, timeout=300)


@pytest.fixture(scope="module")
def checkpoint(tmp_path_factory):
    import torch
    from inversus_b200 import InversusCNNPolicy
    torch.manual_seed(0)
    path = tmp_path_factory.mktemp("ckpt") / "policy.pt"
    torch.save(InversusCNNPolicy().state_dict(), path)
    return str(path)


@pytest.mark.parametrize("args, message", [
    (["--opponent", "medium"], "opponent must be"),
    (["--opponent", "hard", "--episodes_per_env", "0"], "episodes_per_env must be at least 1"),
    (["--opponent", "hard", "--num_envs", "0"], "num_envs must be at least 1"),
    (["--opponent", "@CKPT", "--num_envs", "1"], "head to head needs at least 2 envs"),
    (["--opponent", "hard", "--actions", "argmax"], "invalid choice"),
    (["--opponent", "hard", "--episodes_per_env", "5000000"], "below 2^31"),
])
def test_cli_rejects_bad_arguments(checkpoint, args, message):
    r = _cli("--model", checkpoint, *[checkpoint if a == "@CKPT" else a for a in args])
    assert r.returncode == 2 and message in r.stderr, r.stderr
    assert "Traceback" not in r.stderr


def test_cli_rejects_a_missing_model():
    r = _cli("--model", os.path.join(ROOT, "no_such_policy.pt"), "--opponent", "hard")
    assert r.returncode == 2 and "no such file" in r.stderr and "Traceback" not in r.stderr


def test_cli_fails_cleanly_without_a_device(checkpoint):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    for opp in ("hard", checkpoint):
        r = _cli("--model", checkpoint, "--opponent", opp, "--num_envs", "8", "--episodes_per_env", "1")
        assert r.returncode == 1 and "no CPU fallback" in r.stderr and "Traceback" not in r.stderr, r.stderr
        assert r.stdout == ""


def test_evaluate_rejects_bad_arguments_before_touching_a_device():
    from inversus_b200.evaluate import evaluate
    f = lambda ps: None  # noqa: E731
    with pytest.raises(ValueError, match="opponent"):
        evaluate(f, "medium", 4, 1, seed=0)
    with pytest.raises(ValueError, match="episodes_per_env"):
        evaluate(f, "hard", 4, 0, seed=0)
    with pytest.raises(ValueError, match="head to head"):
        evaluate(f, f, 1, 1, seed=0)
    with pytest.raises(ValueError, match="actions"):
        evaluate(f, "easy", 4, 1, actions="argmax", seed=0)


def test_entry_points_have_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from inversus_b200 import _capi
    lib = _capi.load()
    fake = 1 << 20  # never dereferenced: the device check comes first
    rc = lib.inv_select_actions(fake, 4, fake, 4, 0, 1, 0, 1, fake, None)
    assert rc == _capi.ERR_NO_DEVICE and "no CPU fallback" in _capi.last_error()
    rc = lib.inv_episode_tally(fake, fake, fake, fake, fake, 4, 4, 2, 500, fake, fake, fake, None)
    assert rc == _capi.ERR_NO_DEVICE and "no CPU fallback" in _capi.last_error()
    with pytest.raises(_capi.InversusError, match="no CPU fallback"):
        _capi.check(rc)


def test_evaluate_is_exported_lazily():
    """`inversus_b200.evaluate` is the function, also after the lazy import loaded its submodule."""
    code = ("import inversus_b200, sys; f = inversus_b200.evaluate; "
            "assert 'torch' in sys.modules and callable(f) and f.__name__ == 'evaluate'; "
            "assert inversus_b200.evaluate is f and 'evaluate' in inversus_b200.__all__; print('ok')")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stderr
