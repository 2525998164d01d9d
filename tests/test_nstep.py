"""CPU checks of n-step returns: the restatement the GPU tests hold the sample kernel to (against a naive walk over the
deque), the one-step case, the config key and the refusals that need no GPU."""
import ctypes as C

import numpy as np
import pytest

import replay_oracle as NS
from oracle.replay import RingReplay, zscore_canonical, zscore_stats


def _ring(capacity, n_written, done_logical, seed=0):
    """One agent's ring written ``n_written`` times; ``done_logical``: logical indices (0 = oldest kept) that are done."""
    rng = np.random.default_rng(seed)
    ring = RingReplay(1, capacity, 3)
    total = n_written
    for t in range(total):
        o = rng.integers(-1, 20, (1, 3)).astype(np.float32)
        ring.push(o, np.array([t % 4]), np.array([-float(rng.integers(0, 5000)) * 0.7]), o + 1, np.array([0]))
    size = min(n_written, capacity)
    for j in done_logical:
        ring.done[0, (n_written - size + j) % capacity] = 1
    return ring


def _naive(ring, j, n, gamma, mean, denom):
    """Walk the deque (oldest first) from logical j: the return, the discount and the bootstrap logical index."""
    size = int(min(ring.n_written[0], ring.c))
    order = [(int(ring.n_written[0]) - size + k) % ring.c for k in range(size)]
    ret, k = 0.0, 0
    while True:
        s = order[j + k]
        ret += gamma ** k * ((float(ring.rew[0, s]) - mean) / denom)
        if ring.done[0, s]:
            return ret, 0.0, j + k, True
        if k + 1 == n or j + k + 1 == size:
            return ret, gamma ** (k + 1), j + k, False
        k += 1


CASES = [  # capacity, n_written, done logical indices, n
    (50, 40, [5, 6, 20, 39], 3),        # done inside the window, a return ending exactly on done, the newest row done
    (50, 40, [], 8),                    # no done: only the newest n - 1 rows are truncated
    (30, 77, [0, 13, 28], 5),           # wrapped: returns run past the physical end of the ring
    (4, 11, [2], 8),                    # capacity smaller than n
    (6, 6, [], 16),
    (20, 20, list(range(20)), 4),       # every row done: one-step returns with discount 0
]


@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("cap,nw,dones,n", CASES)
def test_oracle_matches_a_naive_walk_over_the_deque(cap, nw, dones, n, normalize):
    gamma = 0.95
    ring = _ring(cap, nw, dones, seed=cap + nw)
    size = min(nw, cap)
    logical = np.arange(size)
    slots = ring.logical_to_slot(0, logical)
    out = NS.nstep_batch(ring, np.zeros(size, np.int64), slots, n, gamma, normalize)
    mean, denom = zscore_stats(ring.rew[0, slots]) if normalize else (0.0, 1.0)
    for j in range(size):
        ret, disc, last, term = _naive(ring, j, n, gamma, mean, denom)
        assert out["next_slot"][j] == ring.logical_to_slot(0, np.array([last]))[0], f"row {j}: bootstrap row"
        assert out["m"][j] == last - j + 1 and 1 <= out["m"][j] <= min(n, size - j)
        assert out["done"][j] == (1.0 if term else 0.0)
        np.testing.assert_allclose(out["r_hat"][j], np.float32(ret), rtol=2e-6, atol=1e-6, err_msg=f"row {j}: return")
        np.testing.assert_allclose(out["discount"][j], np.float32(disc), rtol=1e-6, err_msg=f"row {j}: discount")
    # the newest n - 1 rows are truncated, never extended past the ring
    assert np.all(out["m"] <= size - logical)


def test_discount_is_the_left_to_right_float64_power():
    ring = _ring(40, 40, [])
    out = NS.nstep_batch(ring, np.zeros(3, np.int64), ring.logical_to_slot(0, np.array([0, 36, 39])), 5, 0.97)
    g = 0.97
    assert out["discount"][0] == np.float32(g * g * g * g * g)
    assert out["discount"][1] == np.float32(g * g * g * g) and out["discount"][2] == np.float32(g)


@pytest.mark.parametrize("n", [0, 1])
@pytest.mark.parametrize("normalize", [True, False])
def test_one_step_is_ring_gather_bit_for_bit(n, normalize):
    ring = _ring(64, 150, [3, 9, 10, 40], seed=5)
    logical = np.random.default_rng(1).integers(0, 64, 48)
    slots = ring.logical_to_slot(0, logical)
    out = NS.nstep_batch(ring, np.zeros(48, np.int64), slots, n, 0.99, normalize)
    _, _, r, _, d = ring.gather(0, logical, normalize_rewards=normalize)
    assert np.array_equal(out["r_hat"], r) and np.array_equal(out["done"], d)
    assert np.array_equal(out["next_slot"], slots) and np.all(out["m"] == 1)
    assert np.array_equal(out["discount"], np.float32(0.99) * (np.float32(1.0) - d))


def test_batch_stats_are_the_canonical_zscore():
    r = -np.random.default_rng(2).integers(0, 5000, 300) * 0.7
    mean, denom = zscore_stats(r)
    assert np.array_equal((r - mean) / denom, zscore_canonical(r))


def test_per_row_discounts_of_gamma_times_one_minus_done_give_the_one_step_learn_step():
    from oracle.dqn import StackedOracle
    rng = np.random.default_rng(3)
    n, b = 2, 16
    s, s2 = rng.integers(-1, 20, (n, b, 89)).astype(np.float32), rng.integers(-1, 20, (n, b, 89)).astype(np.float32)
    a, r = rng.integers(0, 4, (n, b)).astype(np.int32), rng.standard_normal((n, b)).astype(np.float32)
    d = (rng.random((n, b)) < 0.2).astype(np.float32)
    kw = dict(gamma=0.99, learning_rate=5e-4, loss="mse", target_update_frequency=3, seed0=11)
    ns, ws = NS.ReplayStackedOracle(n, 89, [32, 32], 4, **kw), StackedOracle(n, 89, [32, 32], 4, **kw)
    disc = np.float32(0.99) * (np.float32(1.0) - d)
    for _ in range(2):
        x, y = ns.learn_on_batch(s, a, r, s2, d, discounts=disc), ws.learn_on_batch(s, a, r, s2, d)
        assert np.array_equal(x["y"], y["y"]) and np.array_equal(x["loss"], y["loss"])
    # a per-row discount is what the target uses
    z = ns.learn_on_batch(s, a, r, s2, d, discounts=np.zeros((n, b), np.float32))
    assert np.array_equal(z["y"], r)


def test_config_default_and_yaml_key():
    from dmdqn_b200 import train
    from dmdqn_b200.group import DEFAULTS
    assert DEFAULTS["n_step"] == 1
    assert train.load_config()["n_step"] == 1


@pytest.mark.parametrize("n_step", [0, -1, 17])
def test_agent_group_refuses_n_step_outside_1_to_16(n_step):
    from dmdqn_b200.group import AgentGroup
    with pytest.raises(ValueError, match="n_step"):
        AgentGroup(4, {"nn_layers": [64, 64], "n_step": n_step})


def test_hparams_keeps_its_size_with_n_step_in_the_tail_padding():
    from dmdqn_b200 import _native as N
    assert C.sizeof(N.HParams) == 112 and N.HParams.n_step.offset == 108 and N.MAX_NSTEP == 16


@pytest.fixture(scope="module")
def lib():
    from dmdqn_b200 import _native as N
    from dmdqn_b200 import build as B
    B.build()
    return N.lib()


def _hp(n_step):
    from dmdqn_b200 import _native as N
    hp = N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 1000, 0, 1, 1, 0, 1, 0, 0.6, 0.4, 1e-6, 100)
    hp.n_step = n_step
    return hp


@pytest.mark.parametrize("n_step", [17, -1])
def test_native_calls_refuse_n_step_before_launching_anything(lib, n_step):
    from dmdqn_b200 import _native as N
    dims = N.Dims(4, 4, 89, 96, 64, 4, 32, 100)
    nbytes = C.c_size_t()
    N.check(lib.dmdqn_workspace_bytes(C.byref(dims), C.byref(nbytes)))
    ws = (C.c_uint8 * 256)()           # never touched: validation fails before anything is launched
    hp, replay, nets = _hp(n_step), N.Replay(1, 1, 1, 1, 1, 1, None, None), N.Nets(1, 1, 1, 1, 1)
    calls = {
        "learn": lambda: lib.dmdqn_learn(C.byref(dims), C.byref(hp), C.byref(replay), C.byref(nets), C.addressof(ws), None,
                                         None, C.addressof(ws), nbytes.value, None),
        "learn_stages": lambda: lib.dmdqn_learn_stages(C.byref(dims), C.byref(hp), C.byref(replay), C.byref(nets),
                                                       C.addressof(ws), None, None, C.addressof(ws), nbytes.value, 15, None),
        "sample": lambda: lib.dmdqn_sample(C.byref(dims), C.byref(hp), C.byref(replay), C.byref(nets), C.addressof(ws), None,
                                           0, C.addressof(ws), nbytes.value, None),
        "learn_grads": lambda: lib.dmdqn_learn_grads(C.byref(dims), C.byref(hp), C.byref(replay), C.byref(nets),
                                                     C.addressof(ws), None, 32, C.addressof(ws), C.addressof(ws),
                                                     C.addressof(ws), nbytes.value, None),
        "step_host": lambda: lib.dmdqn_step_host(C.byref(dims), C.byref(hp), C.byref(replay), C.byref(nets),
                                                 C.byref(N.StepBlock(256, 0, 16, 32, 48, 64, 80, 89)), C.addressof(ws),
                                                 C.addressof(ws), C.addressof(ws), C.addressof(ws), C.addressof(ws),
                                                 nbytes.value, None),
    }
    for name, call in calls.items():
        assert call() == N.ERR_ARG, name
        assert "n_step" in lib.dmdqn_last_error().decode(), name
