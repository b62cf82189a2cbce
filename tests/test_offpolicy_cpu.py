"""CPU-only: the off-policy oracle's terminal rule, ring-row and uniform-row maps on hand cases, and the C ABI of
rl_explore_mlp / rl_replay_sample_uniform rejecting malformed arguments before anything reaches a device."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import offpolicy as ooff
from oracle import philox as oph


def test_terminal_rule_hand_cases():
    done = np.array([True, True, False, True, False])
    ep_len_before = np.array([0, 4, 4, 998, 999])
    # time limit 5: env 1 reaches length 5 on this step (time limit, not terminal); env 2 too but is not done
    assert ooff.terminal_flags(done, ep_len_before, 5).tolist() == [1, 0, 0, 0, 0]
    assert ooff.terminal_flags(done, ep_len_before, 1000).tolist() == [1, 1, 0, 1, 0]
    assert ooff.terminal_flags(done, ep_len_before, 0).tolist() == [1, 1, 0, 1, 0]      # no time limit


def test_ring_rows_hand_cases():
    assert ooff.ring_rows(0, 0, 4, 10).tolist() == [0, 1, 2, 3]
    assert ooff.ring_rows(0, 2, 4, 10).tolist() == [8, 9, 0, 1]
    assert ooff.ring_rows(7, 1, 3, 10).tolist() == [0, 1, 2]
    # K successive appends of B rows land where one K-step launch puts them
    rows = np.concatenate([ooff.ring_rows(5, t, 3, 11) for t in range(3)])
    assert rows.tolist() == [(5 + i) % 11 for i in range(9)]


def test_uniform_rows_are_the_integer_map():
    k0, k1 = oph.split_seed(9)
    x = oph.philox4x32(np.arange(6, dtype=np.uint32), 4, 0, oph.STREAM_REPLAY, k0, k1)[0]
    for size in (1, 7, 1000, 2 ** 31 - 1):
        rows = ooff.sample_rows(6, 4, size, 9)
        assert rows.tolist() == [(int(v) * size) >> 32 for v in x]
        assert rows.min() >= 0 and rows.max() < size


def test_warmup_actions_are_exact_uniforms():
    a = ooff.uniform_actions(3, np.arange(5, dtype=np.uint32), 2, 6)
    assert a.dtype == np.float32 and a.shape == (5, 6)
    assert (a >= -1).all() and (a < 1).all()
    k0, k1 = oph.split_seed(3)
    w = oph.philox4x32(np.uint32(4), 2, 1, oph.STREAM_ACTION, k0, k1)      # env 4, dims 4..5 = block 1, words 0..1
    assert a[4, 5] == np.float32(2) * oph.u01_24(w[1]) - np.float32(1)


# ---- C ABI argument checks: fake (never dereferenced) pointers, the call must fail before any device work ----------
_P = ctypes.c_void_p(16)


def _explore(dims, head=0, mode=1, K=1, B=4, AD=6, cap=64, pos=0):
    from parl_b200 import _lib
    lib = _lib.load()
    L = len(dims) - 1
    c_dims = (ctypes.c_int * len(dims))(*dims)
    c_layer = (ctypes.c_int * L)(*range(L))
    c_rows = (ctypes.c_int * L)(*dims[1:])
    c_w = (ctypes.c_void_p * L)(*([16] * L))
    rc = lib.rl_explore_mlp(L, c_dims, L, c_layer, c_rows, c_w, None, head, mode, K, B, AD, 0.1, _P, _P, _P, _P, None,
                            None, None, 0, 0, 0, 0, 0.01, 0, _P, _P, _P, _P, _P, cap, pos, None)
    return rc, lib.rl_last_error().decode()


def test_explore_abi_rejects_unsupported_width():
    rc, msg = _explore([17, 600, 64, 6])
    assert rc == -1 and 'width 600' in msg


def test_explore_abi_rejects_launch_larger_than_capacity():
    rc, msg = _explore([17, 256, 256, 6], K=17, B=4, cap=64)
    assert rc == -1 and 'capacity' in msg


def test_explore_abi_rejects_head_mismatch_and_bad_mode():
    rc, msg = _explore([17, 256, 256, 6], head=1, mode=2)
    assert rc == -1 and 'outputs' in msg
    rc, msg = _explore([17, 256, 256, 12], head=1, mode=1)
    assert rc == -1 and 'mode 1' in msg
    rc, msg = _explore([17, 256, 256, 6], mode=3)
    assert rc == -1 and 'mode 3' in msg
    rc, msg = _explore([17, 6])
    assert rc == -1 and 'layers' in msg


def test_explore_wrapper_rejects_cpu_tensors():
    from types import SimpleNamespace
    from parl_b200 import kernels as K
    plan = SimpleNamespace(act=K.ACT_RELU, out_dim=6, dims_list=[17, 256, 256, 6])
    cap = 16
    mem = SimpleNamespace(obs=torch.zeros(cap, 17), action=torch.zeros(cap, 6), reward=torch.zeros(cap, 1),
                          terminal=torch.zeros(cap, 1, dtype=torch.int32), next_obs=torch.zeros(cap, 17),
                          max_size=cap, _curr_pos=0)
    with pytest.raises(RuntimeError, match='CUDA'):
        K.MlpPlan.explore(plan, mem, K.EXPLORE_NOISE, 1, torch.zeros(4, 17), None, 0, 0)
    with pytest.raises(RuntimeError, match='CUDA'):
        K.replay_sample_uniform(mem, 4, torch.ones(1, dtype=torch.int32), torch.zeros(1, dtype=torch.int32), 0)
    with pytest.raises(RuntimeError, match='mode'):
        K.MlpPlan.explore(plan, mem, 7, 1, torch.zeros(4, 17), None, 0, 0)
