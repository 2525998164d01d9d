"""Noisy networks on the GPU (config ``noisy``): the device noise against the float64 restatement (tests/noisy_oracle.py), the
fold bit for bit, the noisy learn step bit for bit against the fold followed by the plain gradient step, the noisy Adam
bit for bit against dmdqn_adam_apply, sigma0 = 0 against a plain group, the semantics against the noisy oracle, act, the
execution orders and the shared-parameter step.  Run on the B200 box: pytest -m gpu"""
import ctypes as C

import numpy as np
import pytest
import torch

import noisy_oracle as O
from oracle.dqn import adam_scalars
from parity_util import NSTEP, PER, RTOL, adam_close, close, draw_words, fill_rings, ulps

pytestmark = pytest.mark.gpu
NOISY = {"noisy": True}
RING = ("obs", "next_obs", "act_ring", "rew_ring", "done_ring", "n_written", "priority", "priority_max")
STATE = ("theta", "theta_tgt", "adam_m", "adam_v", "sigma", "sigma_tgt", "sigma_m", "sigma_v", "learn_step")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _group(n, cap, b, h=64, precision="fp32", a=4, seed=0, **extra):
    from dmdqn_b200.group import AgentGroup
    cfg = {"nn_layers": [h, h], "replay_buffer_size": cap, "batch_size": b, "learning_rate": 5e-4, "gamma": 0.99,
           "target_update_frequency": 3, "precision": precision}
    cfg.update(extra)
    return AgentGroup(n, cfg, action_size=a, seed=seed)


def _fill(grp, n_written, seed):
    fill_rings(grp, n_written, seed=seed, done_rate=0.1)
    grp.act_ring.remainder_(grp.action_size)


def _perturb(grp, seed):
    """Non-zero biases, sigma that differs per element, and a target that differs from the online network."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    for t, s in ((grp.theta, 0.05), (grp.theta_tgt, 0.07)):
        t.add_((grp.theta != 0) * torch.randn(t.shape, device="cuda", generator=gen) * s)
    for t in (grp.sigma, grp.sigma_tgt):
        t.mul_(0.5 + torch.rand(t.shape, device="cuda", generator=gen))


def _keys(grp):
    return [int(k) & ((1 << 64) - 1) for k in grp.key.cpu().tolist()]


def _fold(grp):
    from dmdqn_b200 import _native as N
    N.check(grp.lib.dmdqn_noisy_fold(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.nets), C.byref(grp.noisy_ptrs), _stream()))


def _expected_record(grp, g, t, s):
    return O.noise_record(_keys(grp)[g], t, s, grp.noise_record, grp.state_size, grp.action_size)


def _eps_blocks(grp, g, s, t=None):
    t = int(grp.learn_step[g]) if t is None else t
    return O.eps_block(_expected_record(grp, g, t, s), grp.noise_record, grp.layout, grp.hidden, grp.dueling)


# ------------------------------------------------------------------ 1. noise ------------------------------------------
def test_device_noise_is_the_float64_restatement_within_one_ulp():
    grp = _group(3, 64, 32, h=128, a=3, **NOISY)
    grp.learn_step.copy_(torch.tensor([0, 5, 123456], dtype=torch.int32))
    _fold(grp)
    noise = grp.noise.cpu().numpy()
    off = O.record_offsets(grp.noise_record)
    for g in range(3):
        for s in range(2):
            want = _expected_record(grp, g, int(grp.learn_step[g]), s)
            assert np.all(ulps(noise[g, s], want) <= 1), (g, s)
            assert np.array_equal(noise[g, s] == 0, want == 0), (g, s)             # padding exactly 0, nothing else
            assert np.all(noise[g, s, off[0] + 89:off[1]] == 0) and np.all(noise[g, s, off[5] + 3:off[6]] == 0)
            assert np.all(noise[g, s, off[7] + 1:] == 0)
        assert not np.any((noise[g, 0] == noise[g, 1]) & (noise[g, 0] != 0))     # online and target noise differ
    before = noise.copy()
    grp.learn_step.add_(1)
    _fold(grp)
    after = grp.noise.cpu().numpy()
    assert not np.any((before == after) & (before != 0))                          # step t and t + 1 differ


def test_noise_of_one_group_of_eight_equals_two_groups_of_four():
    big = _group(8, 64, 32, **NOISY)
    halves = [_group(4, 64, 32, seed=4 * k, **NOISY) for k in range(2)]
    for k, hg in enumerate(halves):
        hg.learn_step.copy_(big.learn_step[4 * k:4 * k + 4])
    for grp in [big] + halves:
        _fold(grp)
    assert torch.equal(big.key, torch.cat([hg.key for hg in halves]))
    assert torch.equal(big.noise, torch.cat([hg.noise for hg in halves]))
    assert torch.equal(big.eff, torch.cat([hg.eff for hg in halves]))


# ------------------------------------------------------------------ 2. fold -------------------------------------------
@pytest.mark.parametrize("dueling,a", [(False, 4), (False, 3), (True, 4), (True, 2)])
def test_fold_writes_mu_plus_sigma_times_eps_bit_for_bit(dueling, a):
    grp = _group(3, 64, 32, h=64, a=a, dueling=dueling, **NOISY)
    _perturb(grp, a)
    grp.learn_step.copy_(torch.tensor([2, 0, 77], dtype=torch.int32))
    _fold(grp)
    noise = grp.noise.cpu().numpy()
    for g in range(3):
        for s, mu, sg, eff in ((0, grp.theta, grp.sigma, grp.eff), (1, grp.theta_tgt, grp.sigma_tgt, grp.eff_tgt)):
            e = O.eps_block(noise[g, s], grp.noise_record, grp.layout, grp.hidden, dueling)
            want = O.fold_np(mu[g].cpu().numpy(), sg[g].cpu().numpy(), e)
            assert np.array_equal(eff[g].cpu().numpy(), want), (g, s)


# ------------------------------------------------------------------ 3. plumbing ---------------------------------------
def _learn_grads_noisy(grp, words, grads):
    from dmdqn_b200 import _native as N
    N.check(grp.lib.dmdqn_learn_grads_noisy(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.replay), C.byref(grp.nets),
                                            C.byref(grp.noisy_ptrs), words.data_ptr(), None, grp.batch_size, grads.data_ptr(),
                                            grp.metrics.data_ptr(), grp.workspace.data_ptr(), grp.workspace.numel(), _stream()))


def _learn_grads_on_eff(grp, words, grads):
    from dmdqn_b200 import _native as N
    nets = N.Nets(grp.eff.data_ptr(), grp.eff_tgt.data_ptr(), grp.adam_m.data_ptr(), grp.adam_v.data_ptr(),
                  grp.learn_step.data_ptr())
    N.check(grp.lib.dmdqn_learn_grads(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.replay), C.byref(nets), words.data_ptr(),
                                      None, grp.batch_size, grads.data_ptr(), grp.metrics.data_ptr(), grp.workspace.data_ptr(),
                                      grp.workspace.numel(), _stream()))


def _snapshot(grp):
    return {k: getattr(grp, k).clone() for k in STATE + RING if getattr(grp, k) is not None}


def _restore(grp, snap):
    for k, v in snap.items():
        getattr(grp, k).copy_(v)


@pytest.mark.parametrize("h,precision,extra", [(64, "fp32", {}), (256, "fp32", {}), (256, "tf32x3", {}),
                                               (64, "fp32", dict(**PER, **NSTEP)), (256, "tf32x3", dict(**PER, **NSTEP)),
                                               (64, "fp32", {"dueling": True}), (256, "tf32x3", {"dueling": True, **PER})])
def test_learn_grads_noisy_equals_the_fold_then_plain_learn_grads_on_eff(h, precision, extra):
    n, cap, b = 4, 200, 128
    grp = _group(n, cap, b, h=h, precision=precision, **NOISY, **extra)
    _perturb(grp, h)
    _fill(grp, [cap + 30, 170, cap, 140], seed=h)
    snap = _snapshot(grp)
    words = draw_words(np.random.default_rng(h), n, b)
    outs = []
    for run in (_learn_grads_noisy, None):
        _restore(grp, snap)
        grads = torch.full_like(grp.theta, float("nan"))
        if run is None:
            _fold(grp)
            _learn_grads_on_eff(grp, words, grads)
        else:
            run(grp, words, grads)
        torch.cuda.synchronize()
        dbg = grp.debug_views()
        assert int(dbg["tc_error"][0]) == 0
        outs.append({"metrics": grp.metrics.clone(), "grads": grads, "eff": grp.eff.clone(), "eff_tgt": grp.eff_tgt.clone(),
                     "learn_step": grp.learn_step.clone(), **{k: dbg[k].clone() for k in ("y", "q_all", "q_next", "tq_all")},
                     **({"priority": grp.priority.clone(), "priority_max": grp.priority_max.clone()} if grp.prioritized else {})})
    end = int(grp.layout.b3) + 4 + (grp.hidden + 4 if grp.dueling else 0)      # the range learn_grads writes
    for k in outs[0]:
        sl = (slice(None), slice(0, end)) if k == "grads" else (slice(None),)
        assert torch.equal(outs[0][k][sl], outs[1][k][sl]), k
    assert not outs[0]["grads"][:, :end].isnan().any()
    assert torch.equal(outs[0]["learn_step"], snap["learn_step"] + torch.tensor([1, 1, 1, 1], dtype=torch.int32, device="cuda"))


# ------------------------------------------------------------------ 4. Adam -------------------------------------------
def _adam_apply(grp, nets, grads):
    from dmdqn_b200 import _native as N
    N.check(grp.lib.dmdqn_adam_apply(C.byref(grp.dims), C.byref(grp.hp), C.byref(nets), grads.data_ptr(), grp.workspace.data_ptr(),
                                     grp.workspace.numel(), _stream()))


def _noisy_adam(grp, grads):
    from dmdqn_b200 import _native as N
    N.check(grp.lib.dmdqn_noisy_adam_apply(C.byref(grp.dims), C.byref(grp.hp), C.byref(grp.nets), C.byref(grp.noisy_ptrs),
                                           grads.data_ptr(), grp.workspace.data_ptr(), grp.workspace.numel(), _stream()))


@pytest.mark.parametrize("tau,dueling", [(None, False), (0.05, False), (None, True)])
def test_noisy_adam_equals_adam_apply_on_mu_and_on_sigma_with_g_times_eps(tau, dueling):
    from dmdqn_b200 import _native as N
    n, cap, b = 4, 200, 64
    grp = _group(n, cap, b, tau=tau, dueling=dueling, target_update_frequency=1, **NOISY)
    _perturb(grp, 3)
    _fill(grp, [cap, 30, cap + 9, 150], seed=4)                 # network 1 is inactive
    grp.adam_m.copy_(torch.randn_like(grp.theta) * 1e-3); grp.adam_v.copy_(torch.rand_like(grp.theta) * 1e-6)
    grp.sigma_m.copy_(torch.randn_like(grp.theta) * 1e-3); grp.sigma_v.copy_(torch.rand_like(grp.theta) * 1e-6)
    grp.learn_step.copy_(torch.tensor([3, 4, 5, 6], dtype=torch.int32))
    snap = _snapshot(grp)
    words = draw_words(np.random.default_rng(5), n, b)
    grads = torch.full_like(grp.theta, float("nan"))
    _learn_grads_noisy(grp, words, grads)
    mid = _snapshot(grp)
    _noisy_adam(grp, grads)
    torch.cuda.synchronize()
    got = _snapshot(grp)
    # reference: dmdqn_adam_apply on mu with g, and on sigma's buffers with numpy's g * eps (set 0 at the step's t)
    _restore(grp, mid)
    noise = grp.noise.cpu().numpy()
    g_np = grads.cpu().numpy()
    gs = np.zeros_like(g_np)
    for g in range(n):
        e = O.eps_block(noise[g, 0], grp.noise_record, grp.layout, grp.hidden, dueling)
        gs[g] = (g_np[g] * e).astype(np.float32)
    end = int(grp.layout.b3) + 4 + (grp.hidden + 4 if dueling else 0)
    gs[:, end:] = 0
    g0 = grads.clone(); g0[:, end:] = 0
    _adam_apply(grp, grp.nets, g0)
    _adam_apply(grp, N.Nets(grp.sigma.data_ptr(), grp.sigma_tgt.data_ptr(), grp.sigma_m.data_ptr(), grp.sigma_v.data_ptr(),
                            grp.learn_step.data_ptr()), torch.as_tensor(gs).cuda())
    torch.cuda.synchronize()
    for k in STATE:
        assert torch.equal(got[k], getattr(grp, k)), k
    for k in ("theta", "sigma", "adam_m", "sigma_v", "theta_tgt", "sigma_tgt"):     # the inactive network is untouched
        assert torch.equal(got[k][1], snap[k][1]), k
    assert not torch.equal(got["sigma"], snap["sigma"])
    # a NaN-filled gradient buffer gives the result of a zero-filled one
    _restore(grp, snap)
    grads0 = torch.zeros_like(grp.theta)
    _learn_grads_noisy(grp, words, grads0)
    _noisy_adam(grp, grads0)
    torch.cuda.synchronize()
    for k in STATE:
        assert torch.equal(got[k], getattr(grp, k)), k


# ------------------------------------------------------------------ 5. sigma0 = 0 -------------------------------------
@pytest.mark.parametrize("h,precision", [(64, "fp32"), (256, "tf32x3")])
def test_sigma0_zero_step_equals_a_plain_group(h, precision):
    n, cap, b = 4, 200, 128
    noisy = _group(n, cap, b, h=h, precision=precision, noisy_sigma0=0.0, **NOISY)
    plain = _group(n, cap, b, h=h, precision=precision)
    for grp in (noisy, plain):
        _fill(grp, [cap + 3, cap, 150, 300], seed=8)
    assert torch.equal(noisy.theta, plain.theta) and not noisy.sigma.any()
    words = draw_words(np.random.default_rng(9), n, b)
    mn = noisy.learn(words).clone()
    grads = torch.zeros_like(plain.theta)
    from dmdqn_b200 import _native as N
    N.check(plain.lib.dmdqn_learn_grads(C.byref(plain.dims), C.byref(plain.hp), C.byref(plain.replay), C.byref(plain.nets),
                                        words.data_ptr(), None, b, grads.data_ptr(), plain.metrics.data_ptr(),
                                        plain.workspace.data_ptr(), plain.workspace.numel(), _stream()))
    _adam_apply(plain, plain.nets, grads)
    torch.cuda.synchronize()
    assert torch.equal(mn, plain.metrics)
    for k in ("theta", "theta_tgt", "adam_m", "adam_v", "learn_step"):
        assert torch.equal(getattr(noisy, k), getattr(plain, k)), k
    assert noisy.sigma.any()                    # sigma itself learns away from 0: g_sigma = g * eps


# ------------------------------------------------------------------ 6. semantics --------------------------------------
def _oracle_for(grp, **kw):
    stk = O.NoisyStackedOracle(grp.n_nets, grp.state_size, [grp.hidden] * 2, grp.action_size, gamma=0.99, learning_rate=5e-4,
                               target_update_frequency=3, **kw)
    lists = []
    for which in ("online", "target", "m", "v"):
        per = [grp.get_weights(i, which) for i in range(grp.n_nets)]
        k = len(per[0]) // 2
        lists.append(([torch.stack([p[j] for p in per]) for j in range(k)],
                      [torch.stack([p[k + j] for p in per]) for j in range(k)]))
    (mu, sg), (mt, st), (m, sm), (v, sv) = lists
    stk.set_state(mu, sg, mt, st, m, v, sm, sv)
    stk.learn_step[:] = grp.learn_step.cpu().numpy()
    return stk


def _step_eps(grp, s):
    noise = grp.noise.cpu().numpy()
    per = [O.eps_params(noise[g, s], grp.noise_record, grp.state_size, grp.action_size, grp.dueling) for g in range(grp.n_nets)]
    return [torch.stack([p[k] for p in per]) for k in range(len(per[0]))]


def _oracle_step(grp, stk, rng):
    cap = grp.capacity
    obs, nobs, act = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    metrics = grp.learn(draw_words(rng, grp.n_nets, grp.batch_size)).cpu().numpy()
    dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
    assert int(dbg["tc_error"][0]) == 0
    take = lambda arr, rows: np.stack([arr[g][rows[g] % cap] for g in range(grp.n_nets)])
    out = stk.learn_on_batch(take(obs, dbg["rows"]), take(act, dbg["rows"]), dbg["r_hat"], take(nobs, dbg["next_rows"]), None,
                             _step_eps(grp, 0), _step_eps(grp, 1), discounts=dbg["discount"])
    return metrics, dbg, out


@pytest.mark.parametrize("h,precision", [(64, "fp32"), (128, "fp32"), (256, "fp32"), (512, "fp32"), (256, "tf32x3")])
def test_noisy_learn_matches_the_oracle_on_the_device_noise(h, precision):
    n, cap, b = 3, 200, 128
    grp = _group(n, cap, b, h=h, precision=precision, **NOISY)
    _perturb(grp, h)
    _fill(grp, [cap + 40, 150, cap], seed=h)
    stk = _oracle_for(grp)
    th0 = [[p.clone() for p in ps] for ps in (stk.online, stk.adam_m, stk.adam_v, stk.sigma, stk.sigma_m, stk.sigma_v)]
    t = int(stk.learn_step[0]) + 1
    metrics, dbg, out = _oracle_step(grp, stk, np.random.default_rng(h))
    close(dbg["q_all"], out["q_all"], what="online Q(s)")
    qn = np.sort(out["q_next"], axis=2)
    tie = (qn[..., -1] - qn[..., -2]) < RTOL * np.abs(out["q_next"]).max()
    close(dbg["y"][~tie], out["y"][~tie], what="TD target")
    if tie.any():
        return
    close(metrics[:, 0], out["loss"], what="loss")
    alpha_t, eps_t = adam_scalars(t, 5e-4, "keras")
    for i in range(n):
        got = grp.get_weights(i, "online")
        k = len(got) // 2
        for j in range(2 * k):
            ps, ms, vs = (th0[0], th0[1], th0[2]) if j < k else (th0[3], th0[4], th0[5])
            gk = torch.as_tensor((out["g_mu"] if j < k else out["g_sigma"])[j % k][i])
            adam_close(got[j].numpy(), ps[j % k][i], ms[j % k][i], vs[j % k][i], gk, alpha_t, eps_t, what=f"net {i} param {j}")


@pytest.mark.parametrize("tau", [None, 0.05])
def test_free_running_noisy_trajectory_follows_the_oracle(tau):
    n, cap, b, h = 2, 200, 64, 64
    grp = _group(n, cap, b, h=h, tau=tau, normalize_rewards=False, **NOISY)
    _fill(grp, cap, seed=3)
    grp.rew_ring.mul_(1e-3)
    stk = _oracle_for(grp, tau=tau)
    rng = np.random.default_rng(4)
    for step in range(30):
        metrics, _, out = _oracle_step(grp, stk, rng)
        close(metrics[:, 0], out["loss"], rtol=1e-4, what=f"step {step} loss")
    for i in range(n):
        for which, mu, sg in (("online", stk.online, stk.sigma), ("target", stk.target, stk.sigma_tgt)):
            got = grp.get_weights(i, which)
            for j, ref in enumerate(mu + sg):
                close(got[j].numpy(), ref[i].numpy(), rtol=1e-4, what=f"{which} {j}")


# ------------------------------------------------------------------ 7. act --------------------------------------------
@pytest.mark.parametrize("h,dueling", [(64, False), (128, True), (256, False), (256, True), (512, False)])
def test_act_noisy_equals_plain_act_on_the_folded_block(h, dueling):
    from dmdqn_b200 import _native as N
    n = 6
    grp = _group(n, 64, 32, h=h, dueling=dueling, **NOISY)
    _perturb(grp, h)
    grp.learn_step.copy_(torch.arange(n, dtype=torch.int32) * 7)
    obs = torch.randn((n, 96), device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    a_noisy, q_noisy = grp.act(obs, return_q=True)
    _fold(grp)
    nets = N.Nets(grp.eff.data_ptr(), grp.eff_tgt.data_ptr(), grp.adam_m.data_ptr(), grp.adam_v.data_ptr(), grp.learn_step.data_ptr())
    act = grp.lib.dmdqn_act_dueling if dueling else grp.lib.dmdqn_act
    a_ref = torch.empty_like(a_noisy)
    q_ref = torch.empty_like(q_noisy)
    z = torch.zeros(n, dtype=torch.float64, device="cuda")
    w = torch.zeros(n, dtype=torch.int32, device="cuda")
    N.check(act(C.byref(grp.dims), C.byref(nets), obs.data_ptr(), 96, z.data_ptr(), w.data_ptr(), w.data_ptr(), a_ref.data_ptr(),
                q_ref.data_ptr(), _stream()))
    torch.cuda.synchronize()
    assert torch.equal(q_noisy, q_ref) and torch.equal(a_noisy, a_ref)
    a_mu, q_mu = grp.act(obs, return_q=True, noisy=False)                  # greedy evaluation reads mu
    assert not torch.equal(q_mu, q_noisy)


def test_act_after_a_learn_step_uses_the_next_steps_online_noise():
    grp = _group(3, 200, 64, **NOISY)
    _perturb(grp, 1)
    _fill(grp, 200, seed=2)
    obs = torch.randn((3, 96), device="cuda")
    grp.learn(draw_words(np.random.default_rng(3), 3, 64))
    _, q_act = grp.act(obs, return_q=True)
    snap = _snapshot(grp)
    grads = torch.zeros_like(grp.theta)
    _learn_grads_noisy(grp, draw_words(np.random.default_rng(4), 3, 64), grads)     # folds at the new learn_step
    torch.cuda.synchronize()
    _restore(grp, snap)
    from dmdqn_b200 import _native as N
    nets = N.Nets(grp.eff.data_ptr(), grp.eff_tgt.data_ptr(), 0, 0, grp.learn_step.data_ptr())
    q = torch.empty_like(q_act)
    a = torch.empty((3,), dtype=torch.int32, device="cuda")
    z = torch.zeros(3, dtype=torch.float64, device="cuda")
    w = torch.zeros(3, dtype=torch.int32, device="cuda")
    N.check(grp.lib.dmdqn_act(C.byref(grp.dims), C.byref(nets), obs.data_ptr(), 96, z.data_ptr(), w.data_ptr(), w.data_ptr(),
                              a.data_ptr(), q.data_ptr(), _stream()))
    torch.cuda.synchronize()
    assert torch.equal(q, q_act)


# ------------------------------------------------------------------ 8. execution orders -------------------------------
def test_captured_noisy_learn_equals_plain_learn_and_draws_new_noise_per_replay():
    n, cap, b = 16, 300, 64
    kw = dict(h=256, precision="tf32x3", seed=9, **NOISY)
    a, c = _group(n, cap, b, **kw), _group(n, cap, b, **kw)
    for g in (a, c):
        _fill(g, cap, seed=10)
    replay, draws = c.capture_learn()
    a.learn(draws.clone())
    rng = np.random.default_rng(11)
    noises = []
    for it in range(3):
        w = draw_words(rng, n, b)
        draws.copy_(w)
        mc = replay().clone()
        ma = a.learn(w).clone()
        torch.cuda.synchronize()
        noises.append(c.noise.clone())
        assert torch.equal(ma, mc), it
        for k in STATE:
            assert torch.equal(getattr(a, k), getattr(c, k)), (it, k)
    assert not torch.equal(noises[0], noises[1])


def test_captured_noisy_step_host_equals_step_host():
    n, cap, b = 12, 200, 64
    kw = dict(h=256, precision="tf32x3", seed=5, **NOISY)
    a, c = _group(n, cap, b, **kw), _group(n, cap, b, **kw)
    for g in (a, c):
        _fill(g, cap - 10, seed=12)
    sa, sc = a.make_step_block(), c.make_step_block()
    rng = np.random.default_rng(13)
    replay = None
    for it in range(4):
        vals = {"obs": rng.integers(-1, 20, (n, 89)).astype(np.float32), "next_obs": rng.integers(-1, 20, (n, 89)).astype(np.float32),
                "act": rng.integers(0, 4, n).astype(np.int32), "rew": -rng.random(n) * 100,
                "done": (rng.random(n) < 0.1).astype(np.uint8),
                "draws": rng.integers(0, 2**32, (n, b), dtype=np.uint64).astype(np.uint32).view(np.int32)}
        for blk in (sa, sc):
            for k, v in vals.items():
                blk["host"][k].copy_(torch.as_tensor(v))
        ma = a.step_host(sa)
        if replay is None:
            replay = c.capture_step_host(sc)
            mc = sc["metrics_host"]
        else:
            mc = replay()
        torch.cuda.synchronize()
        assert torch.equal(ma, mc), it
        for k in STATE + ("obs",):
            assert torch.equal(getattr(a, k), getattr(c, k)), (it, k)


def test_one_noisy_group_of_eight_equals_two_groups_of_four():
    n, cap, b = 8, 300, 128
    big = _group(n, cap, b, h=256, precision="tf32x3", **NOISY)
    _fill(big, [cap + 5, cap, 250, 400, 300, 129, 1000, 301], seed=15)
    halves = [_group(4, cap, b, h=256, precision="tf32x3", seed=4 * k, **NOISY) for k in range(2)]
    for k, hg in enumerate(halves):
        for name in RING + STATE:
            if getattr(big, name) is not None:
                getattr(hg, name).copy_(getattr(big, name)[4 * k:4 * k + 4])
        hg.n_written_host[:] = big.n_written_host[4 * k:4 * k + 4]
    rng = np.random.default_rng(16)
    for it in range(3):
        w = draw_words(rng, n, b)
        mb = big.learn(w).clone()
        mh = torch.cat([hg.learn(w[4 * k:4 * k + 4].contiguous()).clone() for k, hg in enumerate(halves)])
        torch.cuda.synchronize()
        assert torch.equal(mb, mh), it
        for name in STATE + ("noise",):
            assert torch.equal(getattr(big, name), torch.cat([getattr(hg, name) for hg in halves])), (it, name)


def test_inactive_networks_keep_every_tensor():
    grp = _group(4, 200, 64, **NOISY)
    _perturb(grp, 6)
    _fill(grp, [200, 10, 200, 63], seed=7)
    snap = _snapshot(grp)
    m = grp.learn(draw_words(np.random.default_rng(8), 4, 64)).cpu().numpy()
    assert list(m[:, 7]) == [1, 0, 1, 0]
    for k in STATE:
        for g in (1, 3):
            assert torch.equal(getattr(grp, k)[g], snap[k][g]), (k, g)
        assert not torch.equal(getattr(grp, k)[0], snap[k][0]) or k in ("theta_tgt", "sigma_tgt"), k


# ------------------------------------------------------------------ 9. shared parameters --------------------------------
def test_shared_noisy_step_world_one_equals_learn_grads_noisy_plus_noisy_adam():
    from dmdqn_b200.parallel import SharedParameterStep
    n, cap, b = 4, 200, 64
    kw = dict(h=64, share_parameters=True, seed=3, **NOISY)
    a, c = _group(n, cap, b, **kw), _group(n, cap, b, **kw)
    for g in (a, c):
        _fill(g, cap, seed=3)
    step = SharedParameterStep.for_group(a)
    assert step.fused_apply is None
    for it in range(3):
        seed = 100 + it
        a._gen.manual_seed(seed); c._gen.manual_seed(seed)
        step.step()
        grads = torch.zeros_like(c.theta)
        _learn_grads_noisy(c, c.draw_words((1, b)), grads)
        _noisy_adam(c, grads)
        c.learn_step_host += 1
        torch.cuda.synchronize()
        for k in STATE:
            assert torch.equal(getattr(a, k), getattr(c, k)), (it, k)


@pytest.mark.parametrize("world", [2, 3])
def test_simulated_ranks_stay_bit_identical(world):
    """Ranks with the same replicas and keys fold the same noise; after the summed block every replica is the same."""
    n, cap, b = 2, 200, 64
    ranks = [_group(n, cap, b, h=64, share_parameters=True, seed=1, **NOISY) for _ in range(world)]
    for r, g in enumerate(ranks):
        _fill(g, cap, seed=20 + r)
    for it in range(2):
        blocks = []
        for g in ranks:
            grads = torch.zeros_like(g.theta)
            _learn_grads_noisy(g, g.draw_words((1, b)), grads)
            blocks.append(grads)
        total = blocks[0].clone()
        for blk in blocks[1:]:
            total += blk
        for g in ranks:
            assert torch.equal(g.noise, ranks[0].noise)
            _noisy_adam(g, total)
        torch.cuda.synchronize()
        for g in ranks[1:]:
            for k in STATE:
                assert torch.equal(getattr(g, k), getattr(ranks[0], k)), (it, k)
