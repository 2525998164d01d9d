"""CPU checks of prioritized replay: the sampler restatement the GPU tests hold the kernel to, the beta schedule and the
importance weights, the weighted learn step, and the refusals that need no GPU."""
import ctypes as C

import numpy as np
import pytest
import torch
from scipy import stats

import replay_oracle as P


def _searchsorted_draw(priority, u):
    """Proportional draw from an exact sequential cumsum: valid when every partial sum is exact (integer priorities)."""
    p = np.asarray(priority, np.float64)
    cs = np.cumsum(p)
    idx = np.searchsorted(cs, u, side="right")
    nz = np.nonzero(p > 0)[0]
    return np.where(idx >= p.shape[0], nz[-1], idx).astype(np.int32)


@pytest.mark.parametrize("cap,zero_frac,seed", [(300, 0.0, 0), (1000, 0.3, 1), (30000, 0.5, 2), (129, 0.9, 3), (128, 0.2, 4)])
def test_integer_priorities_match_searchsorted_on_the_cumsum(cap, zero_frac, seed):
    rng = np.random.default_rng(seed)
    p = rng.integers(1, 50, cap).astype(np.float32)
    p[rng.random(cap) < zero_frac] = 0
    p[-3:] = 0                                         # the clamp must land on the last NON-zero slot
    words = rng.integers(0, 2**32, 256, dtype=np.uint64).astype(np.uint32)
    got = P.prioritized_indices(p, words)
    total = float(p.astype(np.float64).sum())
    assert float(P.chunk_prefixes(p)[-1]) == total
    assert np.array_equal(got, _searchsorted_draw(p, P.stratified_u(total, words)))
    assert np.all(p[got] > 0)
    # u exactly at every chunk edge, exactly at a slot boundary, and at (and past) the total: the clamp
    prefix = P.chunk_prefixes(p)
    cs = np.cumsum(p.astype(np.float64))
    u = np.concatenate([prefix[:-1], cs[::7], [total, total * (1 + 2**-52), 0.0]])
    assert np.array_equal(P.draw_from_u(p, u), _searchsorted_draw(p, u))


def test_zero_priority_slots_are_never_drawn_and_an_all_zero_ring_draws_slot_zero():
    p = np.zeros(500, np.float32)
    p[[3, 260, 261, 499]] = [0.25, 1.5, 0.125, 2.0]
    words = np.arange(0, 2**32, 2**32 // 64, dtype=np.uint64).astype(np.uint32)
    got = P.prioritized_indices(p, words)
    assert set(got.tolist()) <= {3, 260, 261, 499}
    assert np.array_equal(P.prioritized_indices(np.zeros(500, np.float32), words), np.zeros(64, np.int32))


def test_sampler_frequencies_are_proportional_to_priority():
    rng = np.random.default_rng(7)
    cap, b, calls = 200, 64, 400
    p = (rng.random(cap) * 3 + 0.05).astype(np.float32) ** 2
    p[:20] = 0
    hist = np.zeros(cap)
    for _ in range(calls):
        hist += np.bincount(P.prioritized_indices(p, rng.integers(0, 2**32, b, dtype=np.uint64).astype(np.uint32)), minlength=cap)
    assert hist[:20].sum() == 0
    expected = p[20:].astype(np.float64) / p.astype(np.float64).sum() * hist.sum()
    assert stats.chisquare(hist[20:], expected).pvalue > 1e-3


def test_beta_schedule_and_equal_priorities_give_unit_weights():
    assert P.beta_schedule(0, 0.4, 100) == 0.4
    assert P.beta_schedule(50, 0.4, 100) == 0.4 + 0.6 * 50 / 100
    assert P.beta_schedule(100, 0.4, 100) == 1.0 and P.beta_schedule(10**6, 0.4, 100) == 1.0
    assert P.beta_schedule(10**6, 0.4, 0) == 0.4 and P.beta_schedule(5, 0.7, -1) == 0.7
    p = np.full(100, 0.37, np.float32)
    assert np.all(P.is_weights(p, np.arange(100), 0.61) == 1.0)
    p = np.array([1.0, 4.0, 0.5, 2.0], np.float32)
    w = P.is_weights(p, np.array([0, 1, 3, 3]), 0.5)          # slot 2 (the smallest priority) is not drawn
    assert np.array_equal(w, np.array([1.0, 0.5, 2 ** -0.5, 2 ** -0.5], np.float32))


def test_priority_rule_and_ring_push():
    assert P.priority_of(np.array([-2.0, 0.0]), 0.5, 1e-6)[0] == np.float32(np.sqrt(2.0 + 1e-6))
    ring = P.PrioritizedRing(3, 4, 2)
    ring.priority_max[:] = [1.0, 2.0, 3.0]
    z = np.zeros((3, 2), np.float32)
    ring.push(z, np.zeros(3), np.zeros(3), z, np.zeros(3), mask=np.array([1, 0, 1]))
    assert np.array_equal(ring.priority[:, 0], [1.0, 0.0, 3.0])
    ring.update(0, np.array([0, 0]), np.array([3.0, 3.0]), 1.0, 0.0)
    assert ring.priority[0, 0] == 3.0 and ring.priority_max[0] == 3.0


def _oracle_batch(seed, n=2, b=16, h=32, loss="mse"):
    rng = np.random.default_rng(seed)
    s = rng.integers(-1, 20, (n, b, 89)).astype(np.float32)
    s2 = rng.integers(-1, 20, (n, b, 89)).astype(np.float32)
    a = rng.integers(0, 4, (n, b)).astype(np.int32)
    r = rng.standard_normal((n, b)).astype(np.float32)
    d = (rng.random((n, b)) < 0.1).astype(np.float32)
    kw = dict(gamma=0.99, learning_rate=5e-4, loss=loss, target_update_frequency=3, seed0=11)
    return (s, a, r, s2, d), P.ReplayStackedOracle(n, 89, [h, h], 4, **kw), P.StackedOracle(n, 89, [h, h], 4, **kw)


@pytest.mark.parametrize("loss", ["mse", "huber"])
def test_weighted_gradient_is_the_gradient_of_the_weighted_loss(loss):
    batch, wstk, _ = _oracle_batch(1, loss=loss)
    w = np.random.default_rng(2).uniform(0.1, 1.0, (2, 16)).astype(np.float32)
    params = [p.clone().requires_grad_(True) for p in wstk.online]
    out = wstk.learn_on_batch(*batch, is_weights=w)
    # independent restatement: dL/dq = w_i * (the unweighted per-row gradient), back-propagated through the network
    s, a = torch.as_tensor(batch[0]), torch.as_tensor(batch[1]).long()
    pred = torch.gather(P.StackedOracle.forward(params, s), 2, a[..., None])[..., 0]
    _, g = P.loss_and_grad(pred.detach(), torch.as_tensor(out["y"]), loss)
    ref = torch.autograd.grad(pred, params, grad_outputs=torch.as_tensor(w) * g)
    for got, r in zip(out["grads"], ref):
        np.testing.assert_allclose(got, r.numpy(), rtol=1e-5, atol=1e-6 * float(r.abs().max()))
    assert np.allclose(out["loss"], (w * P.loss_and_grad(pred.detach(), torch.as_tensor(out["y"]), loss)[0].numpy()).mean(1))
    assert np.array_equal(out["delta"], pred.detach().numpy() - out["y"])


@pytest.mark.parametrize("loss", ["mse", "huber"])
def test_unit_weights_give_the_unweighted_step_exactly(loss):
    batch, wstk, stk = _oracle_batch(3, loss=loss)
    for _ in range(2):
        a = wstk.learn_on_batch(*batch, is_weights=np.ones((2, 16), np.float32))
        b = stk.learn_on_batch(*batch)
        assert np.array_equal(a["loss"], b["loss"])
        for x, y in zip(a["grads"], b["grads"]):
            assert np.array_equal(x, y)
    for name in ("online", "target", "adam_m", "adam_v"):
        for x, y in zip(getattr(wstk, name), getattr(stk, name)):
            assert torch.equal(x, y)


def test_prioritized_with_shared_parameters_is_rejected_before_the_library_loads():
    from dmdqn_b200.group import AgentGroup
    with pytest.raises(ValueError, match="independent networks"):
        AgentGroup(4, {"nn_layers": [64, 64], "share_parameters": True, "sample_mode": "prioritized"})


def test_config_file_lists_the_prioritized_keys():
    from dmdqn_b200 import train
    from dmdqn_b200.group import DEFAULTS
    cfg = train.load_config()
    assert cfg["sample_mode"] == "fisher_yates"
    for k in ("per_alpha", "per_beta", "per_beta_steps", "per_eps"):
        assert cfg[k] == DEFAULTS[k]


@pytest.fixture(scope="module")
def lib():
    from dmdqn_b200 import _native as N
    from dmdqn_b200 import build as B
    B.build()
    return N.lib()


def _learn_call(lib, dims, replay, sample_mode=3):
    from dmdqn_b200 import _native as N
    nbytes = C.c_size_t()
    N.check(lib.dmdqn_workspace_bytes(C.byref(dims), C.byref(nbytes)))
    ws = (C.c_uint8 * 256)()           # never touched: validation fails before anything is launched
    hp = N.HParams(0.99, 5e-4, 0.9, 0.999, 1e-7, -1.0, 1000, 0, 1, 1, 0, sample_mode, 0, 0.6, 0.4, 1e-6, 100)
    nets = N.Nets(1, 1, 1, 1, 1)
    return lib.dmdqn_learn(C.byref(dims), C.byref(hp), C.byref(replay), C.byref(nets), C.addressof(ws), None, None,
                           C.addressof(ws), nbytes.value, None)


def test_prioritized_mode_without_a_priority_array_is_rejected_with_a_message(lib):
    from dmdqn_b200 import _native as N
    dims = N.Dims(4, 4, 89, 96, 64, 4, 32, 100)
    rc = _learn_call(lib, dims, N.Replay(1, 1, 1, 1, 1, 1, None, None))
    assert rc == N.ERR_ARG and "NULL priority pointer" in lib.dmdqn_last_error().decode()
    shared = N.Dims(4, 1, 89, 96, 64, 4, 32, 100)
    rc = _learn_call(lib, shared, N.Replay(1, 1, 1, 1, 1, 1, 1, 1))
    assert rc == N.ERR_ARG and "independent networks" in lib.dmdqn_last_error().decode()
    assert _learn_call(lib, dims, N.Replay(1, 1, 1, 1, 1, 1, 1, 1), sample_mode=4) == N.ERR_ARG


def test_abi_version_and_mode_constants(lib):
    from dmdqn_b200 import _native as N
    assert lib.dmdqn_abi_version() == 3 and N.SAMPLE["prioritized"] == 3
    assert N.HParams.per_alpha.offset % 8 == 0 and N.Replay.priority.offset == 6 * C.sizeof(C.c_void_p)
