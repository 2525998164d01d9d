"""Prioritized replay on the GPU (sample_mode "prioritized") against tests/per_oracle.py: the push rule, the drawn slots
(bit-exact), the importance weights, the weighted learn step and its priority update, equivalence with the uniform path
when every weight is 1, and the execution orders that must not change a bit.  Run on the B200 box: pytest -m gpu"""
import ctypes as C

import numpy as np
import pytest
import torch

import per_oracle as P
from parity_util import RTOL, adam_close, close

pytestmark = pytest.mark.gpu


def _group(n, cap, b, h=64, precision="fp32", seed=0, **extra):
    from dmdqn_b200.group import AgentGroup
    cfg = {"nn_layers": [h, h], "replay_buffer_size": cap, "batch_size": b, "learning_rate": 5e-4, "gamma": 0.99,
           "target_update_frequency": 3, "precision": precision, "sample_mode": "prioritized"}
    cfg.update(extra)
    return AgentGroup(n, cfg, seed=seed)


def _fill(grp, n_written, seed, priorities=True):
    """Ring contents straight into the device tensors; n_written per agent; non-integer priorities on the written slots."""
    n, cap = grp.n_agents, grp.capacity
    gen = torch.Generator(device="cuda").manual_seed(seed)
    grp.obs[:, :, :89] = torch.randint(-1, 20, (n, cap, 89), device="cuda", generator=gen).float()
    grp.next_obs[:, :, :89] = torch.randint(-1, 20, (n, cap, 89), device="cuda", generator=gen).float()
    grp.act_ring.copy_(torch.randint(0, 4, (n, cap), device="cuda", generator=gen).int())
    grp.rew_ring.copy_(-torch.randint(0, 5000, (n, cap), device="cuda", generator=gen).double() * 0.7)
    grp.done_ring.copy_((torch.rand((n, cap), device="cuda", generator=gen) < 0.05).to(torch.uint8))
    nw = np.broadcast_to(np.asarray(n_written, np.int64), (n,)).copy()
    grp.n_written.copy_(torch.as_tensor(nw)); grp.n_written_host[:] = nw
    if priorities and grp.priority is not None:
        size = torch.as_tensor(np.minimum(nw, cap), device="cuda")
        written = torch.arange(cap, device="cuda")[None, :] < size[:, None]
        p = torch.rand((n, cap), device="cuda", generator=gen) * 2 + 0.01
        grp.priority.copy_(torch.where(written, p, torch.zeros_like(p)))
        grp.priority_max.copy_(grp.priority.max(1).values)


def _words(rng, n, b):
    return torch.as_tensor(rng.integers(0, 2**32, (n, b), dtype=np.uint64).astype(np.uint32).view(np.int32)).cuda()


def _ulps(a, b):
    return np.abs(np.asarray(a, np.float32).view(np.int32).astype(np.int64) - np.asarray(b, np.float32).view(np.int32))


def _copy_state(dst, src, sl=slice(None)):
    for name in ("obs", "next_obs", "act_ring", "rew_ring", "done_ring", "n_written", "priority", "priority_max",
                 "theta", "theta_tgt", "adam_m", "adam_v", "learn_step"):
        getattr(dst, name).copy_(getattr(src, name)[sl])
    dst.n_written_host[:] = src.n_written_host[sl]
    dst.learn_step_host[:] = src.learn_step_host[sl]


# ------------------------------------------------------------------ 1. push ---------------------------------------------
def test_push_gives_new_slots_the_maximum_priority():
    n, cap = 4, 5
    grp = _group(n, cap, 2)
    ring = P.PrioritizedRing(n, cap, 89)
    rng = np.random.default_rng(0)
    for t in range(13):
        if t in (3, 8):                                # the ring's maximum moves (as the learn step would move it)
            pm = rng.uniform(0.5, 4.0, n).astype(np.float32)
            grp.priority_max.copy_(torch.as_tensor(pm)); ring.priority_max[:] = pm
        mask = (rng.random(n) < 0.7).astype(np.uint8)
        s = rng.integers(-1, 20, (n, 89)).astype(np.float32)
        a, r, dn = rng.integers(0, 4, n).astype(np.int32), rng.random(n), np.zeros(n, bool)
        grp.push(s, a, r, s, dn, mask=mask); ring.push(s, a, r, s, dn, mask=mask)
        assert np.array_equal(grp.priority.cpu().numpy(), ring.priority), f"push {t}"
    assert np.array_equal(grp.n_written.cpu().numpy(), ring.n_written) and ring.n_written.max() > cap   # wrapped around
    assert np.array_equal(grp.priority_max.cpu().numpy(), ring.priority_max)


# ------------------------------------------------------------------ 2. sampling -----------------------------------------
def test_sampling_is_bit_exact_against_the_oracle():
    from oracle import replay as R
    n, cap, b = 16, 30000, 256
    grp = _group(n, cap, b, per_beta=0.45)
    n_written = np.array([256, 300, 1000, 5000, 12345, 20000, 29999, 30000, 30001, 45678, 60000, 256 + 128, 777, 4096,
                          29000, 100000])
    _fill(grp, n_written, seed=1)
    rng = np.random.default_rng(2)
    pr = grp.priority.cpu().numpy()
    rew = grp.rew_ring.cpu().numpy()
    for it in range(3):
        words = _words(rng, n, b)
        grp.sample(words)
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        w = words.cpu().numpy().view(np.uint32)
        for g in range(n):
            slots = P.prioritized_indices(pr[g], w[g])
            assert np.array_equal(dbg["rows"][g], g * cap + slots), f"call {it} agent {g}: drawn slots differ"
            assert np.all(slots < min(n_written[g], cap))
            ref = P.is_weights(pr[g], slots, 0.45)     # sample() does not advance learn_step: beta_t = beta0
            assert _ulps(dbg["is_weights"][g], ref).max() <= 2, f"call {it} agent {g}: importance weights"
            assert np.array_equal(dbg["r_hat"][g], R.zscore_canonical(rew[g, slots]).astype(np.float32))


# ------------------------------------------------------------------ 3. frequencies --------------------------------------
def test_device_frequencies_are_proportional_to_priority():
    from scipy import stats
    n, cap, b, calls = 2, 300, 64, 300
    grp = _group(n, cap, b)
    _fill(grp, cap, seed=3)
    grp.priority[:, :40] = 0
    grp.priority[1, 100:110] *= 20
    pr = grp.priority.cpu().numpy().astype(np.float64)
    rng = np.random.default_rng(4)
    hist = np.zeros((n, cap))
    for _ in range(calls):
        grp.sample(_words(rng, n, b))
        rows = grp.debug_views()["rows"].cpu().numpy()
        for g in range(n):
            hist[g] += np.bincount(rows[g] - g * cap, minlength=cap)
    for g in range(n):
        assert hist[g, :40].sum() == 0
        expected = pr[g, 40:] / pr[g].sum() * hist[g].sum()
        assert stats.chisquare(hist[g, 40:], expected).pvalue > 1e-4


# ------------------------------------------------------------------ 4. learn parity -------------------------------------
def _weighted_branch_gradients(params, states, actions, y, w, loss_kind, mask1, mask2):
    """Float64 gradients of mean_i(w_i * term_i) on the ReLU branch the kernel took (its relu' masks)."""
    w1, b1, w2, b2, w3, b3 = (np.asarray(p, np.float64) for p in params)
    x = np.asarray(states, np.float64)
    b = x.shape[1]
    h1 = np.maximum(np.einsum("nbd,ndh->nbh", x, w1) + b1[:, None, :], 0)
    h2 = np.maximum(np.einsum("nbh,nhk->nbk", h1, w2) + b2[:, None, :], 0)
    q = np.einsum("nbh,nha->nba", h2, w3) + b3[:, None, :]
    a = np.asarray(actions, np.int64)
    e = np.take_along_axis(q, a[..., None], 2)[..., 0] - np.asarray(y, np.float64)
    gcoef = (2 * e / b if loss_kind == "mse" else np.clip(e, -1, 1) / b) * np.asarray(w, np.float64)
    dq = np.zeros_like(q)
    np.put_along_axis(dq, a[..., None], gcoef[..., None], 2)
    dh2 = np.einsum("nba,nha->nbh", dq, w3) * np.asarray(mask2, bool)
    dh1 = np.einsum("nbk,nhk->nbh", dh2, w2) * np.asarray(mask1, bool)
    grads = [np.einsum("nbd,nbh->ndh", x, dh1), dh1.sum(1), np.einsum("nbh,nbk->nhk", h1, dh2), dh2.sum(1),
             np.einsum("nbh,nba->nha", h2, dq), dq.sum(1)]
    return [g.astype(np.float32) for g in grads]


@pytest.mark.parametrize("h,precision,loss", [(64, "fp32", "mse"), (64, "fp32", "huber"), (256, "fp32", "mse"),
                                              (256, "tf32x3", "mse"), (256, "tf32x3", "huber")])
def test_learn_matches_the_weighted_oracle(h, precision, loss):
    from oracle import replay as R
    from oracle.dqn import adam_scalars
    n, cap, b, alpha, eps, beta0, beta_steps = 3, 200, 128, 0.6, 1e-6, 0.4, 4
    grp = _group(n, cap, b, h=h, precision=precision, loss=loss, per_alpha=alpha, per_eps=eps, per_beta=beta0,
                 per_beta_steps=beta_steps)
    rng = np.random.default_rng(h + len(loss))
    stk = P.WeightedStackedOracle(n, 89, [h, h], 4, gamma=0.99, learning_rate=5e-4, loss=loss, target_update_frequency=3,
                                  seed0=50)
    for k in (1, 3, 5):
        stk.online[k] += torch.as_tensor(rng.standard_normal(stk.online[k].shape).astype(np.float32)) * 0.05
        stk.target[k].copy_(stk.online[k])

    def load():
        for i in range(n):
            for which, src in (("online", stk.online), ("target", stk.target), ("m", stk.adam_m), ("v", stk.adam_v)):
                grp.set_weights(i, [p[i] for p in src], which)
    load()
    _fill(grp, [cap + 40, 150, cap], seed=h)
    obs, nobs = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89]
    act, rew, done = grp.act_ring.cpu().numpy(), grp.rew_ring.cpu().numpy(), grp.done_ring.cpu().numpy()
    for step in range(6):
        words = _words(rng, n, b)
        pr0, pmax0 = grp.priority.cpu().numpy(), grp.priority_max.cpu().numpy()
        metrics = grp.learn(words).cpu().numpy()
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        assert int(dbg["tc_error"][0]) == 0
        t = int(stk.learn_step[0]) + 1
        w = words.cpu().numpy().view(np.uint32)
        slots = dbg["rows"] - np.arange(n)[:, None] * cap
        beta = P.beta_schedule(t, beta0, beta_steps)
        for g in range(n):
            assert np.array_equal(slots[g], P.prioritized_indices(pr0[g], w[g])), f"step {step} agent {g}: slots"
            assert _ulps(dbg["is_weights"][g], P.is_weights(pr0[g], slots[g], beta)).max() <= 2
        isw = dbg["is_weights"]
        take = lambda a: np.stack([a[g, slots[g]] for g in range(n)])
        S, A_, S2, D = take(obs), take(act), take(nobs), take(done).astype(np.float32)
        Rw = np.stack([R.zscore_canonical(rew[g, slots[g]]) for g in range(n)]).astype(np.float32)
        assert np.array_equal(dbg["r_hat"], Rw)
        th0 = [p.clone() for p in stk.online]; m0 = [p.clone() for p in stk.adam_m]; v0 = [p.clone() for p in stk.adam_v]
        out = stk.learn_on_batch(S, A_, Rw, S2, D, is_weights=isw)
        qn = np.sort(out["q_next"], axis=2)
        tie = (qn[..., -1] - qn[..., -2]) < RTOL * np.abs(out["q_next"]).max()
        assert tie.mean() < 0.01
        close(dbg["q_all"], out["q_all"], what=f"step {step} online Q(s)")
        close(dbg["y"][~tie], out["y"][~tie], what=f"step {step} TD target")
        # the new priorities come from the device's own q(s)[a] and y, within 1 ulp; nothing else moves
        delta = np.take_along_axis(dbg["q_all"], A_[..., None].astype(np.int64), 2)[..., 0] - dbg["y"]
        pr1, pmax1 = grp.priority.cpu().numpy(), grp.priority_max.cpu().numpy()
        for g in range(n):
            pref = P.priority_of(delta[g], alpha, eps)
            assert _ulps(pr1[g, slots[g]], pref).max() <= 1, f"step {step} agent {g}: priorities"
            untouched = np.ones(cap, bool); untouched[slots[g]] = False
            assert np.array_equal(pr1[g, untouched], pr0[g, untouched])
            assert pmax1[g] == max(pmax0[g], pr1[g, slots[g]].max())
        if tie.any():
            load()
            continue
        close(metrics[:, 0], out["loss"], what=f"step {step} weighted loss")
        g64 = _weighted_branch_gradients([p.numpy() for p in th0], S, A_, out["y"], isw, loss, dbg["dh1"] != 0,
                                         dbg["dh2"] != 0)
        alpha_t, eps_t = adam_scalars(t, 5e-4, "keras")
        for i in range(n):
            got, gm, gv = grp.get_weights(i, "online"), grp.get_weights(i, "m"), grp.get_weights(i, "v")
            for k in range(6):
                gk = torch.as_tensor(g64[k][i])
                adam_close(got[k].numpy(), th0[k][i], m0[k][i], v0[k][i], gk, alpha_t, eps_t, what=f"step {step} net {i} theta[{k}]")
                close(gm[k].numpy(), (m0[k][i] + (gk - m0[k][i]) * np.float32(0.1)).numpy(), what=f"step {step} net {i} m[{k}]")
                close(gv[k].numpy(), (v0[k][i] + (gk * gk - v0[k][i]) * np.float32(0.001)).numpy(), rtol=2 * RTOL,
                      what=f"step {step} net {i} v[{k}]")
        load()                                          # keep the trajectories together: later steps test the kernel


# ------------------------------------------------------------------ 5. equivalence with uniform -------------------------
@pytest.mark.parametrize("h,precision", [(64, "fp32"), (256, "tf32x3")])
def test_alpha_zero_equals_the_uniform_path_on_the_same_rows(h, precision):
    n, cap, b = 5, 300, 64
    per = _group(n, cap, b, h=h, precision=precision, seed=4, per_alpha=0.0)
    uni = _group(n, cap, b, h=h, precision=precision, seed=4, sample_mode="indices")
    for g in (per, uni):
        _fill(g, [cap + 17, cap, 200, 64, 1000], seed=6, priorities=False)
    per.priority.copy_((torch.arange(cap, device="cuda")[None, :] < torch.as_tensor(per.sizes_host(), device="cuda")[:, None]).float())
    rng = np.random.default_rng(7)
    nw = per.n_written_host.copy()
    for step in range(4):
        mp = per.learn(_words(rng, n, b)).clone()
        dbg = per.debug_views()
        assert torch.all(dbg["is_weights"] == 1.0)
        slots = dbg["rows"].cpu().numpy() - np.arange(n)[:, None] * cap
        size = np.minimum(nw, cap)
        logical = (slots - (nw - size)[:, None]) % cap
        mu = uni.learn(logical.astype(np.int32)).clone()
        torch.cuda.synchronize()
        assert torch.equal(mp, mu), f"step {step}: metrics differ"
        for name in ("theta", "theta_tgt", "adam_m", "adam_v", "learn_step"):
            assert torch.equal(getattr(per, name), getattr(uni, name)), f"step {step}: {name} differs"
        written = torch.as_tensor(per.sizes_host(), device="cuda")[:, None] > torch.arange(cap, device="cuda")[None, :]
        assert torch.all(per.priority[written] == 1.0) and torch.all(per.priority[~written] == 0.0)


# ------------------------------------------------------------------ 6. execution order ----------------------------------
def test_chained_step_equals_stage_by_stage_step():
    from dmdqn_b200 import _native as N
    n, cap, b = 40, 160, 128
    a, c = _group(n, cap, b, h=256, precision="tf32x3", seed=2), _group(n, cap, b, h=256, precision="tf32x3", seed=2)
    for g in (a, c):
        _fill(g, cap + 3, seed=8)
    rng = np.random.default_rng(9)
    for it in range(4):
        w = _words(rng, n, b)
        ma = a.learn(w).clone()
        for stage in (1, 2, 4, 8):
            N.check(c.lib.dmdqn_learn_stages(C.byref(c.dims), C.byref(c.hp), C.byref(c.replay), C.byref(c.nets), w.data_ptr(),
                                             None, c.metrics.data_ptr(), c.workspace.data_ptr(), c.workspace.numel(), stage,
                                             torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert torch.equal(ma, c.metrics), f"step {it}: metrics differ"
        for name in ("theta", "theta_tgt", "adam_m", "adam_v", "priority", "priority_max"):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name} differs"


def test_captured_learn_equals_plain_learn_while_beta_anneals():
    n, cap, b = 16, 300, 64
    kw = dict(h=256, precision="tf32x3", seed=9, per_beta_steps=3)
    a, c = _group(n, cap, b, **kw), _group(n, cap, b, **kw)
    for g in (a, c):
        _fill(g, cap, seed=10)
    replay, draws = c.capture_learn()
    a.learn(draws.clone())                             # the capture's warm-up step, on a
    rng = np.random.default_rng(11)
    for it in range(5):                                # beta_t = 0.6, 0.8, 1.0, 1.0, ...: the graph reads it on the device
        w = _words(rng, n, b)
        draws.copy_(w)
        mc = replay().clone()
        ma = a.learn(w).clone()
        torch.cuda.synchronize()
        assert torch.equal(ma, mc), f"step {it}: metrics differ"
        assert torch.equal(a.debug_views()["is_weights"], c.debug_views()["is_weights"])
        for name in ("theta", "theta_tgt", "adam_m", "adam_v", "priority", "priority_max", "learn_step"):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name} differs"


def test_captured_step_host_equals_step_host():
    n, cap, b = 12, 200, 64
    a, c = _group(n, cap, b, h=256, precision="tf32x3", seed=5), _group(n, cap, b, h=256, precision="tf32x3", seed=5)
    for g in (a, c):
        _fill(g, cap, seed=12)
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
        assert torch.equal(ma, mc), f"step {it}: metrics differ"
        for name in ("theta", "theta_tgt", "adam_m", "adam_v", "priority", "priority_max", "obs"):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name} differs"


def test_one_group_of_eight_equals_two_groups_of_four():
    n, cap, b = 8, 300, 128
    big = _group(n, cap, b, h=256, precision="tf32x3", seed=14)
    _fill(big, [cap + 5, cap, 250, 400, 300, 129, 1000, 301], seed=15)
    halves = [_group(4, cap, b, h=256, precision="tf32x3", seed=99) for _ in range(2)]
    for k, hg in enumerate(halves):
        _copy_state(hg, big, slice(4 * k, 4 * k + 4))
    rng = np.random.default_rng(16)
    for it in range(4):
        w = _words(rng, n, b)
        mb = big.learn(w).clone()
        mh = torch.cat([hg.learn(w[4 * k:4 * k + 4].contiguous()).clone() for k, hg in enumerate(halves)])
        torch.cuda.synchronize()
        assert torch.equal(mb, mh), f"step {it}: metrics differ"
        for name in ("theta", "theta_tgt", "adam_m", "adam_v", "priority", "priority_max"):
            assert torch.equal(getattr(big, name), torch.cat([getattr(hg, name) for hg in halves])), f"step {it}: {name}"


# ------------------------------------------------------------------ 7. duplicates ---------------------------------------
@pytest.mark.parametrize("h,precision", [(64, "fp32"), (256, "tf32x3")])
def test_a_slot_drawn_twice_keeps_the_priority_of_either_row(h, precision):
    n, cap, b, alpha, eps = 2, 200, 64, 0.7, 1e-6
    grp = _group(n, cap, b, h=h, precision=precision, per_alpha=alpha, per_eps=eps)
    _fill(grp, cap, seed=17)
    grp.priority[:, 10] = 1e4                          # slot 10 carries most of the mass: drawn many times per batch
    grp.priority[:, 11] = 5e3
    grp.learn(_words(np.random.default_rng(18), n, b))
    dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
    pr = grp.priority.cpu().numpy()
    act = np.stack([grp.act_ring.cpu().numpy()[g, dbg["rows"][g] - g * cap] for g in range(n)])
    delta = np.take_along_axis(dbg["q_all"], act[..., None].astype(np.int64), 2)[..., 0] - dbg["y"]
    for g in range(n):
        slots = dbg["rows"][g] - g * cap
        for s in (10, 11):
            rows = np.nonzero(slots == s)[0]
            assert rows.size >= 2
            assert np.all(delta[g, rows] == delta[g, rows[0]])      # one transition, one TD error
            assert _ulps(pr[g, s], P.priority_of(delta[g, rows[:1]], alpha, eps)).max() <= 1


# ------------------------------------------------------------------ the training loop -----------------------------------
@pytest.mark.parametrize("mode", ["batched", "per_agent"])
def test_train_loop_runs_prioritized_from_the_config_alone(mode):
    """train_agents needs nothing but the config: both call patterns learn with prioritized replay, and the learn steps
    move the priorities of the slots they drew."""
    from dmdqn_b200.train import PRESETS, train_agents
    cfg = dict(PRESETS["shipped_train_py"])
    cfg.update(max_sim_time=600.0, backend="fake", grid_rows=3, grid_cols=3, fake_traci_seed=11, batch_size=16,
               nn_layers=[64, 64], precision="auto", sample_mode="prioritized", per_beta_steps=10)
    history, agents, group = train_agents(cfg, episodes=1, mode=mode, seed=3, learn=True)
    assert group.prioritized and group.priority.shape == (9, group.capacity)
    t = len(history)
    assert t > 16 and np.all(group.learn_step.cpu().numpy() == t - 15)      # one learn step per step once 16 are stored
    assert any(h["total_loss"] != 0 for h in history)
    pr = group.priority.cpu().numpy()
    assert np.all(pr[:, :t] > 0) and np.all(pr[:, t:] == 0)
    assert np.any(pr[:, :t] != 1.0)                                            # priorities from TD errors, not only the push rule
    assert int(group.debug_views()["tc_error"][0]) == 0
