"""Host arithmetic of the overlapped step for ping-pong rollouts of two passes per CTA (``csrc/planner.cu``
``overlap_schedule``, exported by ``nlc_debug_overlap_plan``; no device): the first pass's samples are encoded before the
fork, and only the last steps of the last pass's samples beside the rollout."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    from neurallaplacecontrol_b200 import _lib

    return _lib.load()


def _plan(lib, K, T, nx=6, S=17):
    out = (C.c_longlong * 8)()
    assert lib.nlc_debug_overlap_plan(K, T, nx, S, out) == 0
    overlap, pp, sms, passes, k1, split, total, beside = tuple(out)
    return dict(overlap=overlap, pp=pp, sms=sms, passes=passes, k1=k1, split=split, total=total, beside=beside)


def _old(lib, K, T, nx=6, S=17):
    fn = lib.nlc_debug_overlap_schedule
    fn.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_longlong)]
    fn.restype = C.c_int
    out = (C.c_longlong * 4)()
    assert fn(K, T, nx, S, out) == 0
    return tuple(out)


def test_config4_runs_its_last_pass_beside_the_encoder_tail(lib):
    s = _plan(lib, 65536, 50)
    assert (s["overlap"], s["pp"], s["sms"], s["passes"], s["k1"]) == (1, 1, 128, 2, 32768)
    # the last pass's 32768 samples are 256 tiles per step; its last n (and a part of one more) steps are encoded beside the
    # rollout
    assert s["total"] == 50 * 256 and s["beside"] * 256 <= s["total"] - s["split"] < (s["beside"] + 1) * 256
    assert 5 <= s["beside"] <= 8


def test_two_pass_limit_is_140_rollout_sms(lib):
    # 560 tiles: 140 CTAs x 2 passes leave the encoder 8 SMs; 561 tiles would need 141
    s = _plan(lib, 560 * 128, 50)
    assert s["overlap"] == 1 and s["sms"] == 140 and s["passes"] == 2
    s = _plan(lib, 561 * 128, 50)
    assert s["overlap"] == 0


def test_ragged_two_pass_plans(lib):
    # acrobot 40001 x 20: 313 tiles on 79 CTAs; the last pass covers samples [79 * 256, 40001)
    s = _plan(lib, 40001, 20)
    assert (s["overlap"], s["pp"], s["sms"], s["passes"], s["k1"]) == (1, 1, 79, 2, 79 * 256)
    sub = (40001 - 79 * 256 + 127) // 128
    assert s["total"] == 20 * sub and 0 < s["split"] < s["total"] and s["beside"] == (s["total"] - s["split"]) // sub
    # cartpole 50000 x 9: 391 tiles on 98 CTAs
    s = _plan(lib, 50000, 9, nx=5)
    assert (s["overlap"], s["sms"], s["passes"], s["k1"]) == (1, 98, 2, 98 * 256)
    assert s["total"] == 9 * ((50000 - 98 * 256 + 127) // 128)


@pytest.mark.parametrize("K,T,nx,S", [(8192, 50, 6, 17), (16384, 50, 6, 17), (32768, 50, 6, 17), (88 * 128, 50, 6, 17),
                                      (89 * 128, 50, 6, 17), (1000, 20, 3, 17), (8192, 30, 5, 17), (16384, 50, 6, 33),
                                      (280 * 128, 50, 6, 17)])
def test_one_pass_sizes_match_the_schedule_entry_point(lib, K, T, nx, S):
    s = _plan(lib, K, T, nx, S)
    assert s["passes"] == 1 and s["k1"] == 0
    assert (s["pp"], s["sms"], s["split"], s["total"]) == _old(lib, K, T, nx, S)
