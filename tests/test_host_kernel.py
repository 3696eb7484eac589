"""The product's OWN game logic on the CPU: the device functions of csrc/inversus_kernels.cuh
(load_env / rl_step / rl_reset / debug_phase / build_row / store_env, everything except the kernel
shell) and the canonical-state conversions of inv_export_state / inv_import_state are compiled for
the host through tests/host_kernel/host_shim.h and

  * replayed against every committed golden fixture of the live Python reference -- the same
    bit-exact bar as the GPU parity tests, but runnable without a GPU, with the state read back
    through the product's own export,
  * driven through the reference's own engine unit tests and the state import/export checks, and
  * run under AddressSanitizer + UBSan on a random rollout that also round-trips every env through
    export and import (compute-sanitizer is closed on the GPU pool, so this is the memory-safety
    check of the shared logic: bullet slots, tile words, observation rows, state conversion).

This is a test harness, not a fallback: nothing in the product can reach it (INV_HOST_BUILD is
defined only by tests/host_kernel/harness.cpp)."""
import os
import subprocess

import numpy as np
import pytest

from backends import HostKernelBackend, check_state_import_export
from golden.scenarios import SCENARIOS, compare, run_scenario

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_kernel_logic_on_host_reproduces_reference_fixture(name):
    sc = SCENARIOS[name]
    gold = dict(np.load(os.path.join(GOLD, f"{name}.npz")))
    rec = run_scenario(HostKernelBackend(sc), sc)
    compare(rec, gold, float_rtol=1e-6, what=name)
    assert np.array_equal(rec["reward_f32"], gold["reward_f32"])
    assert np.array_equal(rec["episode_return"], gold["episode_return"])


def test_kernel_logic_under_address_and_ub_sanitizers(tmp_path):
    hk = os.path.join(HERE, "host_kernel")
    exe = str(tmp_path / "hk_san")
    cmd = ["g++", "-O1", "-g", "-std=c++17", "-ffp-contract=off", "-Wno-unknown-pragmas", "-fsanitize=address,undefined",
           "-fno-sanitize-recover=all", "-DHK_STANDALONE", "-I", hk, "-o", exe, os.path.join(hk, "harness.cpp")]
    b = subprocess.run(cmd, capture_output=True, text=True)
    if b.returncode != 0 and ("asan" in b.stderr.lower() or "sanitize" in b.stderr.lower()):
        pytest.skip("sanitizer runtime not available: " + b.stderr[-200:])
    assert b.returncode == 0, b.stderr[-2000:]
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, ASAN_OPTIONS="detect_leaks=0"))
    assert r.returncode == 0, r.stdout[-1000:] + r.stderr[-3000:]
    assert "sanitizer run ok" in r.stdout


def test_state_import_export_roundtrip_and_validation_on_host():
    b = HostKernelBackend(dict(n=64, mode="dummy", difficulty="hard", max_steps=500, seed=1))
    b.reset(None)
    check_state_import_export(b.export_state, b.import_state)


import reference_kat as K  # noqa: E402


@pytest.mark.parametrize("name", K.ALL_KATS)
def test_reference_unit_tests_through_the_kernel_logic_on_host(name):
    """The reference's own unit tests (tests/reference_kat.py) against the product's engine
    functions compiled for the host -- the CPU twin of tests/test_cuda_reference_kat.py."""
    from engine_facade import HostKernelEngine
    getattr(K, name)(lambda w, h: HostKernelEngine(w, h))


FRESH = {
    "host_hard": dict(mode="dummy", difficulty="hard", max_steps=500, n=512, T=600, seed=301, actions="uniform", draws="philox", resets="auto"),
    "host_easy": dict(mode="dummy", difficulty="easy", max_steps=120, n=256, T=300, seed=302, actions="shooty", draws="philox", resets="auto"),
    "host_selfplay": dict(mode="selfplay", difficulty="hard", max_steps=200, n=256, T=300, seed=303, actions="shooty", draws="philox", resets="auto"),
    "host_table": dict(mode="dummy", difficulty="hard", max_steps=90, n=200, T=200, seed=305, actions="charge", draws="table", resets="manual"),
}


@pytest.mark.parametrize("name", sorted(FRESH))
def test_kernel_logic_on_host_matches_oracle_on_fresh_seeds(name):
    from backends import OracleBackend
    sc = FRESH[name]
    want = run_scenario(OracleBackend(sc, nthreads=4), sc, record_obs=(sc["n"] <= 256))
    got = run_scenario(HostKernelBackend(sc), sc, record_obs=(sc["n"] <= 256))
    compare(got, want, float_rtol=1e-6, what=name)
    assert np.array_equal(got["reward_f32"], want["reward_f32"])
    assert np.array_equal(got["episode_return"], want["episode_return"])
