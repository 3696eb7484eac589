"""Every handle-free compute entry point of the C ABI reports its own failures in inv_last_error():
without an sm_100 device it fails with INV_ERR_NO_DEVICE ("no CPU fallback"), and on a B200 an
invalid argument fails with INV_ERR_INVALID_ARG and a message naming the entry point. Both checks
first leave an unrelated message behind (a failed inv_create) so that a stale text cannot pass."""
import ctypes as C

import pytest

from inversus_b200 import _capi

FAKE = 1 << 20  # a 16-byte-aligned address that is never dereferenced: every call here fails first


def _poison(lib):
    handle = C.c_void_p()
    assert lib.inv_create(C.byref(_capi.Config(n_envs=0)), C.byref(handle)) == _capi.ERR_INVALID_ARG
    assert _capi.last_error().startswith("inv_create:")


def _valid_looking_calls(lib):
    f = FAKE
    return {
        "inv_ln_relu_fwd": lambda: lib.inv_ln_relu_fwd(f, None, None, f, f, 4, 4800, 32, 1e-5, f, f, f, None),
        "inv_ln_relu_bwd": lambda: lib.inv_ln_relu_bwd(f, f, None, None, f, f, f, f, 4, 4800, 32, f, f, f, None, f, None),
        "inv_transpose_cast": lambda: lib.inv_transpose_cast(f, 1, 64, f, 0, 64, 4, 8, 8, None),
        "inv_encode_fwd": lambda: lib.inv_encode_fwd(f, 4, 4, 0, f, f, f, f, 1e-5, f, None, f, f, None),
        "inv_encode_bwd": lambda: lib.inv_encode_bwd(f, 4, 4, 0, *[f] * 12, None),
        "inv_conv3x3_wgrad": lambda: lib.inv_conv3x3_wgrad(f, f, 4, 128, 128, f, f, None),
        "inv_gae": lambda: lib.inv_gae(f, f, f, None, 0.99, 0.95, 8, 4, f, f, None),
        "inv_select_actions": lambda: lib.inv_select_actions(f, 4, f, 4, 0, 1, 0, 1, f, None),
        "inv_episode_tally": lambda: lib.inv_episode_tally(f, f, f, f, f, 4, 4, 1, 500, f, f, f, None),
    }


# one invalid argument per entry point, the rest as above
def _invalid_calls(lib):
    f = FAKE
    return {
        "inv_ln_relu_fwd": lambda: lib.inv_ln_relu_fwd(f, None, None, f, f, 4, 4804, 32, 1e-5, f, f, f, None),
        "inv_ln_relu_bwd": lambda: lib.inv_ln_relu_bwd(f, f, None, None, f, f, f, f, 4, 4804, 32, f, f, f, None, f, None),
        "inv_transpose_cast": lambda: lib.inv_transpose_cast(f, 1, 64, f, 1, 64, 4, 8, 8, None),
        "inv_encode_fwd": lambda: lib.inv_encode_fwd(f, 4, 4, 2, f, f, f, f, 1e-5, f, None, f, f, None),
        "inv_encode_bwd": lambda: lib.inv_encode_bwd(f, 4, 4, 2, *[f] * 12, None),
        "inv_conv3x3_wgrad": lambda: lib.inv_conv3x3_wgrad(f + 8, f, 4, 128, 128, f, f, None),
        "inv_gae": lambda: lib.inv_gae(f, f, f, None, 0.99, 0.95, -1, 4, f, f, None),
        "inv_select_actions": lambda: lib.inv_select_actions(f, 4, f, 4, 0, 1, 2, 1, f, None),
        "inv_episode_tally": lambda: lib.inv_episode_tally(f, f, f, f, f, 4, 4, 0, 500, f, f, f, None),
    }


NAMES = sorted(_valid_looking_calls(None))


@pytest.mark.parametrize("name", NAMES)
def test_no_device_error_names_the_entry_point(name):
    lib = _capi.load()
    if lib.inv_device_count() > 0:
        pytest.skip("a GPU is present")
    _poison(lib)
    rc = _valid_looking_calls(lib)[name]()
    msg = _capi.last_error()
    assert rc == _capi.ERR_NO_DEVICE, (rc, msg)
    assert msg.startswith(name + ":") and "no CPU fallback" in msg, msg
    with pytest.raises(_capi.InversusError, match="no CPU fallback"):
        _capi.check(rc)


def test_no_device_even_for_empty_work():
    lib = _capi.load()
    if lib.inv_device_count() > 0:
        pytest.skip("a GPU is present")
    _poison(lib)
    assert lib.inv_gae(FAKE, FAKE, FAKE, None, 0.99, 0.95, 0, 4, FAKE, FAKE, None) == _capi.ERR_NO_DEVICE
    assert lib.inv_transpose_cast(FAKE, 1, 64, FAKE, 0, 64, 0, 8, 8, None) == _capi.ERR_NO_DEVICE
    assert _capi.last_error().startswith("inv_transpose_cast:")


def test_size_queries_answer_anywhere():
    lib = _capi.load()
    assert lib.inv_ln_relu_partials(4800) > 0
    assert lib.inv_encode_partials_floats() > 0
    for cin, cout in ((128, 128), (64, 128), (32, 64)):
        assert lib.inv_conv3x3_wgrad_scratch_floats(cin, cout) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_invalid_argument_error_names_the_entry_point(name):
    lib = _capi.load()
    _poison(lib)
    rc = _invalid_calls(lib)[name]()
    msg = _capi.last_error()
    assert rc == _capi.ERR_INVALID_ARG, (rc, msg)
    assert msg.startswith(name + ":") and len(msg) > len(name) + 2, msg
    with pytest.raises(ValueError, match=name):
        _capi.check(rc)
