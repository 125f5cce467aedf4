"""CPU: auvrrt_plan_group is the one rule for the planner a batch runs (the rule launch_plan applies to group 0), and it
needs no device; without a device the _dev entries of the planning step's device end fail loudly."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def auvrrt():
    from auvrrt import build
    build.build()
    import auvrrt
    return auvrrt


def _group(api, Q, with_path, **kw):
    return api.plan_group(api.plan_params(64, **kw), Q, with_path)


@pytest.mark.parametrize("group", [32, 16, 8])
def test_explicit_groups_pass_through(auvrrt, group):
    api = auvrrt.api
    for Q in (0, 1, 32767, 32768, 1 << 20):
        for with_path in (False, True):
            for mode in (0, 1, 2, 3):
                assert _group(api, Q, with_path, group=group, mode=mode) == group


def test_explicit_thread_per_tree(auvrrt):
    api = auvrrt.api
    for Q in (1, 32768):
        for mode in (0, 1, 2):
            assert _group(api, Q, False, group=1, mode=mode) == 1
            # (launch_plan refuses a path with group 1; the rule itself names the planner)
            assert _group(api, Q, True, group=1, mode=mode) == 1
    with pytest.raises(auvrrt.AuvrrtError, match="mode 3"):
        _group(api, 100, False, group=1, mode=3)


def test_group_zero_picks_thread_per_tree_only_for_large_pathless_batches(auvrrt):
    api = auvrrt.api
    for mode in (0, 1, 2):
        assert _group(api, 32767, False, mode=mode) == 32
        assert _group(api, 32768, False, mode=mode) == 1
        assert _group(api, 1 << 20, False, mode=mode) == 1
        assert _group(api, 32768, True, mode=mode) == 32
        assert _group(api, 0, False, mode=mode) == 32
    for Q in (1, 32768, 1 << 20):
        for with_path in (False, True):
            assert _group(api, Q, with_path, mode=3) == 32


@pytest.mark.parametrize("bad", [2, 4, 7, 33, 64, -1])
def test_bad_groups(auvrrt, bad):
    api, L = auvrrt.api, auvrrt.lib()
    assert L.auvrrt_plan_group(C.byref(api.plan_params(64, group=bad)), 100, 0) == -1
    assert b"group" in L.auvrrt_last_error()
    with pytest.raises(auvrrt.AuvrrtError, match="group"):
        _group(api, 100, False, group=bad)
    assert L.auvrrt_plan_group(None, 100, 0) == -1


def test_dev_entries_without_a_device(auvrrt):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L, api = auvrrt.lib(), auvrrt.api
    pp = api.plan_params(64, group=32, path_cap=16)
    assert L.auvrrt_plan_best_dev(None, 0, None, 1, None, None, None) == 2
    assert b"no CUDA device" in L.auvrrt_last_error()
    assert L.auvrrt_materialize_dev(None, None, None, None, None, 0, None, 1, C.byref(pp), 0, None, None, None) == 2
    assert b"no CUDA device" in L.auvrrt_last_error()
