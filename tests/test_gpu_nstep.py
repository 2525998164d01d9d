"""n-step returns on the GPU (n_step > 1) against tests/nstep_oracle.py: the sampled returns, discounts and bootstrap rows
(bit-exact, every sample mode), the unchanged one-step path, learn parity, prioritized replay and shared parameters with
n-step targets, and the execution orders that must not change a bit.  Run on the B200 box: pytest -m gpu"""
import ctypes as C

import numpy as np
import pytest
import torch

import nstep_oracle as NS
import per_oracle as P
from oracle import replay as R
from oracle.replay import RingReplay
from parity_util import RTOL, adam_close, close

pytestmark = pytest.mark.gpu


def _group(n, cap, b, h=64, precision="fp32", seed=0, **extra):
    from dmdqn_b200.group import AgentGroup
    cfg = {"nn_layers": [h, h], "replay_buffer_size": cap, "batch_size": b, "learning_rate": 5e-4, "gamma": 0.99,
           "target_update_frequency": 3, "precision": precision, "n_step": 3}
    cfg.update(extra)
    return AgentGroup(n, cfg, seed=seed)


def _fill(grp, n_written, seed, done_rate=0.05):
    """Ring contents straight into the device tensors (about 5 % done); n_written per agent; priorities on written slots."""
    n, cap = grp.n_agents, grp.capacity
    gen = torch.Generator(device="cuda").manual_seed(seed)
    grp.obs[:, :, :89] = torch.randint(-1, 20, (n, cap, 89), device="cuda", generator=gen).float()
    grp.next_obs[:, :, :89] = torch.randint(-1, 20, (n, cap, 89), device="cuda", generator=gen).float()
    grp.act_ring.copy_(torch.randint(0, 4, (n, cap), device="cuda", generator=gen).int())
    grp.rew_ring.copy_(-torch.randint(0, 5000, (n, cap), device="cuda", generator=gen).double() * 0.7)
    grp.done_ring.copy_((torch.rand((n, cap), device="cuda", generator=gen) < done_rate).to(torch.uint8))
    nw = np.broadcast_to(np.asarray(n_written, np.int64), (n,)).copy()
    grp.n_written.copy_(torch.as_tensor(nw)); grp.n_written_host[:] = nw
    if grp.priority is not None:
        size = torch.as_tensor(np.minimum(nw, cap), device="cuda")
        written = torch.arange(cap, device="cuda")[None, :] < size[:, None]
        p = torch.rand((n, cap), device="cuda", generator=gen) * 2 + 0.01
        grp.priority.copy_(torch.where(written, p, torch.zeros_like(p)))
        grp.priority_max.copy_(grp.priority.max(1).values)


def _host_ring(grp):
    """The group's rewards, done flags and fill levels as an oracle ring (observations are compared separately)."""
    ring = RingReplay(grp.n_agents, grp.capacity, 1)
    ring.rew = grp.rew_ring.cpu().numpy()
    ring.done = grp.done_ring.cpu().numpy()
    ring.n_written = grp.n_written.cpu().numpy().astype(np.int64)
    return ring


def _words(rng, n, b):
    return torch.as_tensor(rng.integers(0, 2**32, (n, b), dtype=np.uint64).astype(np.uint32).view(np.int32)).cuda()


def _ulps(a, b):
    return np.abs(np.asarray(a, np.float32).view(np.int32).astype(np.int64) - np.asarray(b, np.float32).view(np.int32))


def _check_against_oracle(grp, ring, dbg, n, normalize=True, what=""):
    """rows -> the oracle's returns, discounts, terminal flags and bootstrap rows, bit for bit; returns the oracle per net."""
    cap, outs = grp.capacity, []
    for g in range(grp.n_nets):
        rows = dbg["rows"][g]
        out = NS.nstep_batch(ring, rows // cap, rows % cap, n, 0.99, normalize)
        assert np.array_equal(dbg["next_rows"][g], (rows // cap) * cap + out["next_slot"]), f"{what} net {g}: bootstrap rows"
        assert np.array_equal(dbg["r_hat"][g], out["r_hat"]), f"{what} net {g}: returns"
        assert np.array_equal(dbg["discount"][g], out["discount"]), f"{what} net {g}: discounts"
        outs.append(out)
    return outs


# ------------------------------------------------------------------ 1. sampling -----------------------------------------
N_WRITTEN = np.array([256, 300, 1000, 5000, 12345, 20000, 29999, 30000, 30001, 45678, 60000, 384, 777, 4096, 29000, 100000])


@pytest.mark.parametrize("n", [3, 8])
@pytest.mark.parametrize("mode", ["fisher_yates", "replacement", "indices", "prioritized"])
def test_sampling_is_bit_exact_against_the_oracle(mode, n):
    cap, b = 30000, 256
    grp = _group(16, cap, b, n_step=n, sample_mode=mode)
    _fill(grp, N_WRITTEN, seed=1)
    ring = _host_ring(grp)
    size = np.minimum(N_WRITTEN, cap)
    nobs = grp.next_obs.cpu().numpy()[..., :89]
    pr = grp.priority.cpu().numpy() if grp.priority is not None else None
    rng = np.random.default_rng(2)
    for it in range(2):
        if mode == "indices":                          # the newest rows of every ring, then random ones
            draws = np.stack([np.concatenate([size[g] - 1 - np.arange(16), rng.integers(0, size[g], b - 16)])
                              for g in range(16)]).astype(np.int32)
            dev = torch.as_tensor(draws).cuda()
        else:
            dev = _words(rng, 16, b)
            draws = dev.cpu().numpy().view(np.uint32)
        states, actions, rewards, next_states, dones, active = grp.sample(dev)
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        for g in range(16):
            if mode == "prioritized":
                slots = P.prioritized_indices(pr[g], draws[g])
            else:
                logical = {"fisher_yates": lambda: R.fisher_yates_indices(draws[g], size[g]),
                           "replacement": lambda: R.replacement_indices(draws[g], size[g]),
                           "indices": lambda: draws[g]}[mode]()
                slots = ring.logical_to_slot(g, logical)
            assert np.array_equal(dbg["rows"][g], g * cap + slots), f"{mode} call {it} agent {g}: rows"
        outs = _check_against_oracle(grp, ring, dbg, n, what=f"{mode} call {it}")
        assert any(o["m"].min() < n for o in outs) and all(o["m"].max() <= n for o in outs)
        dones_ref = np.stack([o["done"] for o in outs])
        assert np.array_equal(dones.cpu().numpy(), dones_ref) and np.array_equal(rewards.cpu().numpy(), dbg["r_hat"])
        nref = np.stack([nobs[g, dbg["next_rows"][g] - g * cap] for g in range(16)])
        assert np.array_equal(next_states.cpu().numpy(), nref), f"{mode} call {it}: gathered next states"
        assert np.all(active.cpu().numpy() == 1)
        if mode == "indices":                          # the newest row of every ring bootstraps from itself
            assert np.all(dbg["next_rows"][:, 0] == dbg["rows"][:, 0])


# ------------------------------------------------------------------ 2. one-step path ------------------------------------
@pytest.mark.parametrize("precision,h", [("fp32", 64), ("tf32x3", 256)])
@pytest.mark.parametrize("mode", ["fisher_yates", "prioritized"])
def test_n_step_one_and_zero_are_the_one_step_path_bit_for_bit(precision, h, mode):
    from dmdqn_b200.group import AgentGroup
    n, cap, b = 6, 300, 64
    base = {"nn_layers": [h, h], "replay_buffer_size": cap, "batch_size": b, "learning_rate": 5e-4, "gamma": 0.99,
            "target_update_frequency": 3, "precision": precision, "sample_mode": mode}
    plain = AgentGroup(n, base, seed=4)
    one = AgentGroup(n, dict(base, n_step=1), seed=4)
    zero = AgentGroup(n, dict(base, n_step=1), seed=4)
    zero.hp.n_step = 0                                 # what a zero-initialised C caller passes
    groups = (plain, one, zero)
    for grp in groups:
        _fill(grp, [cap + 17, cap, 200, 64, 1000, 150], seed=6, done_rate=0.2)
    rng = np.random.default_rng(7)
    for step in range(4):
        w = _words(rng, n, b)
        ms = [grp.learn(w).clone() for grp in groups]
        torch.cuda.synchronize()
        dbg = [grp.debug_views() for grp in groups]
        for k in (1, 2):
            assert torch.equal(ms[0], ms[k]), f"step {step} group {k}: metrics"
            assert torch.equal(dbg[0]["y"], dbg[k]["y"]) and torch.equal(dbg[0]["rows"], dbg[k]["next_rows"])
            for name in ("theta", "theta_tgt", "adam_m", "adam_v", "priority", "priority_max"):
                a, c = getattr(plain, name), getattr(groups[k], name)
                assert (a is None and c is None) or torch.equal(a, c), f"step {step} group {k}: {name}"


# ------------------------------------------------------------------ 3. learn parity -------------------------------------
@pytest.mark.parametrize("h,precision,loss,double_dqn,mode", [
    (64, "fp32", "mse", True, "fisher_yates"), (64, "fp32", "huber", False, "fisher_yates"),
    (256, "fp32", "mse", False, "fisher_yates"), (256, "fp32", "huber", True, "fisher_yates"),
    (256, "tf32x3", "mse", True, "fisher_yates"), (256, "tf32x3", "huber", False, "fisher_yates"),
    (64, "fp32", "mse", True, "prioritized"), (256, "tf32x3", "huber", True, "prioritized")])
def test_learn_matches_the_n_step_oracle(h, precision, loss, double_dqn, mode):
    from oracle.dqn import adam_scalars
    from test_gpu_prioritized import _weighted_branch_gradients
    n, cap, b, alpha, eps = 3, 200, 128, 0.6, 1e-6
    grp = _group(n, cap, b, h=h, precision=precision, loss=loss, double_dqn=double_dqn, sample_mode=mode,
                 per_alpha=alpha, per_eps=eps, per_beta=1.0)
    rng = np.random.default_rng(h + len(loss) + double_dqn)
    stk = NS.NStepStackedOracle(n, 89, [h, h], 4, gamma=0.99, learning_rate=5e-4, loss=loss, target_update_frequency=3,
                                double_dqn=double_dqn, seed0=50)
    for k in (1, 3, 5):
        stk.online[k] += torch.as_tensor(rng.standard_normal(stk.online[k].shape).astype(np.float32)) * 0.05
        stk.target[k].copy_(stk.online[k])

    def load():
        for i in range(n):
            for which, src in (("online", stk.online), ("target", stk.target), ("m", stk.adam_m), ("v", stk.adam_v)):
                grp.set_weights(i, [p[i] for p in src], which)
    load()
    _fill(grp, [cap + 40, 150, cap], seed=h, done_rate=0.1)
    ring = _host_ring(grp)
    obs, nobs, act = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    for step in range(5):
        pr0 = grp.priority.cpu().numpy() if grp.priority is not None else None
        metrics = grp.learn(_words(rng, n, b)).cpu().numpy()
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        assert int(dbg["tc_error"][0]) == 0
        outs = _check_against_oracle(grp, ring, dbg, 3, what=f"step {step}")
        t = int(stk.learn_step[0]) + 1
        slots, nslots = dbg["rows"] % cap, dbg["next_rows"] % cap
        take = lambda a, s: np.stack([a[g, s[g]] for g in range(n)])
        S, A_, S2 = take(obs, slots), take(act, slots), take(nobs, nslots)
        Rn = np.stack([o["r_hat"] for o in outs])
        D = np.stack([o["done"] for o in outs])
        disc = np.stack([o["discount"] for o in outs])
        isw = dbg["is_weights"] if mode == "prioritized" else None
        th0 = [p.clone() for p in stk.online]; m0 = [p.clone() for p in stk.adam_m]; v0 = [p.clone() for p in stk.adam_v]
        out = stk.learn_on_batch(S, A_, Rn, S2, D, is_weights=isw, discounts=disc)
        qn = np.sort(out["q_next"], axis=2)
        tie = (qn[..., -1] - qn[..., -2]) < RTOL * np.abs(out["q_next"]).max()
        assert tie.mean() < 0.01
        close(dbg["q_all"], out["q_all"], what=f"step {step} online Q(s)")
        close(dbg["y"][~tie], out["y"][~tie], what=f"step {step} TD target")
        if mode == "prioritized":                      # the row's priority from its n-step TD error, within 1 ulp
            delta = np.take_along_axis(dbg["q_all"], A_[..., None].astype(np.int64), 2)[..., 0] - dbg["y"]
            pr1 = grp.priority.cpu().numpy()
            for g in range(n):
                assert _ulps(pr1[g, slots[g]], P.priority_of(delta[g], alpha, eps)).max() <= 1, f"step {step} agent {g}"
                untouched = np.ones(cap, bool); untouched[slots[g]] = False
                assert np.array_equal(pr1[g, untouched], pr0[g, untouched])
        if tie.any():
            load()
            continue
        close(metrics[:, 0], out["loss"], what=f"step {step} loss")
        w = isw if isw is not None else np.ones((n, b), np.float32)
        g64 = _weighted_branch_gradients([p.numpy() for p in th0], S, A_, out["y"], w, loss, dbg["dh1"] != 0,
                                         dbg["dh2"] != 0)
        alpha_t, eps_t = adam_scalars(t, 5e-4, "keras")
        for i in range(n):
            got = grp.get_weights(i, "online")
            for k in range(6):
                adam_close(got[k].numpy(), th0[k][i], m0[k][i], v0[k][i], torch.as_tensor(g64[k][i]), alpha_t, eps_t,
                           what=f"step {step} net {i} theta[{k}]")
        load()                                          # keep the trajectories together: later steps test the kernel


# ------------------------------------------------------------------ 4. shared parameters --------------------------------
def test_shared_parameters_keep_every_lookahead_in_its_own_ring():
    n, cap, b = 6, 120, 256
    grp = _group(n, cap, b, share_parameters=True, n_step=5)
    _fill(grp, cap + 33, seed=20, done_rate=0.05)
    ring = _host_ring(grp)
    stk = NS.NStepStackedOracle(1, 89, [64, 64], 4, gamma=0.99, learning_rate=5e-4, loss="mse", target_update_frequency=3,
                                seed0=7)
    grp.set_weights(0, [p[0] for p in stk.online], "online"); grp.set_weights(0, [p[0] for p in stk.target], "target")
    obs, nobs, act = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    rng = np.random.default_rng(21)
    w = _words(rng, 1, b)
    grp.learn(w)
    dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
    rows, nrows = dbg["rows"][0], dbg["next_rows"][0]
    logical = R.fisher_yates_indices(w.cpu().numpy().view(np.uint32)[0], cap * n)
    agents = logical // cap
    assert np.array_equal(rows // cap, agents) and np.array_equal(nrows // cap, agents), "a lookahead crossed rings"
    assert np.array_equal(rows % cap, [ring.logical_to_slot(a, np.array([j]))[0] for a, j in zip(agents, logical % cap)])
    (o,) = _check_against_oracle(grp, ring, dbg, 5, what="shared")
    assert o["m"].min() < 5 and o["m"].max() == 5
    out = stk.learn_on_batch(obs[agents, rows % cap][None], act[agents, rows % cap][None], o["r_hat"][None],
                             nobs[agents, nrows % cap][None], o["done"][None], discounts=o["discount"][None])
    close(dbg["y"], out["y"], what="shared TD target")
    close(dbg["q_all"], out["q_all"], what="shared online Q(s)")


# ------------------------------------------------------------------ 5. execution order ----------------------------------
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
        for name in ("theta", "theta_tgt", "adam_m", "adam_v"):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name} differs"


def test_captured_learn_equals_plain_learn():
    n, cap, b = 16, 300, 64
    kw = dict(h=256, precision="tf32x3", seed=9)
    a, c = _group(n, cap, b, **kw), _group(n, cap, b, **kw)
    for g in (a, c):
        _fill(g, cap, seed=10)
    replay, draws = c.capture_learn()
    a.learn(draws.clone())                             # the capture's warm-up step, on a
    rng = np.random.default_rng(11)
    for it in range(4):
        w = _words(rng, n, b)
        draws.copy_(w)
        mc = replay().clone()
        ma = a.learn(w).clone()
        torch.cuda.synchronize()
        assert torch.equal(ma, mc), f"step {it}: metrics differ"
        for name in ("theta", "theta_tgt", "adam_m", "adam_v", "learn_step"):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name} differs"


def test_captured_step_host_equals_step_host():
    n, cap, b = 12, 200, 64
    a, c = _group(n, cap, b, h=256, precision="tf32x3", seed=5), _group(n, cap, b, h=256, precision="tf32x3", seed=5)
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
        assert torch.equal(ma, mc), f"step {it}: metrics differ"
        for name in ("theta", "theta_tgt", "adam_m", "adam_v", "obs", "done_ring"):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name} differs"


def test_one_group_of_eight_equals_two_groups_of_four():
    n, cap, b = 8, 300, 128
    big = _group(n, cap, b, h=256, precision="tf32x3", seed=14)
    _fill(big, [cap + 5, cap, 250, 400, 300, 129, 1000, 301], seed=15)
    halves = [_group(4, cap, b, h=256, precision="tf32x3", seed=99) for _ in range(2)]
    for k, hg in enumerate(halves):
        sl = slice(4 * k, 4 * k + 4)
        for name in ("obs", "next_obs", "act_ring", "rew_ring", "done_ring", "n_written", "theta", "theta_tgt", "adam_m",
                     "adam_v", "learn_step"):
            getattr(hg, name).copy_(getattr(big, name)[sl])
        hg.n_written_host[:] = big.n_written_host[sl]
        hg.learn_step_host[:] = big.learn_step_host[sl]
    rng = np.random.default_rng(16)
    for it in range(4):
        w = _words(rng, n, b)
        mb = big.learn(w).clone()
        mh = torch.cat([hg.learn(w[4 * k:4 * k + 4].contiguous()).clone() for k, hg in enumerate(halves)])
        torch.cuda.synchronize()
        assert torch.equal(mb, mh), f"step {it}: metrics differ"
        for name in ("theta", "theta_tgt", "adam_m", "adam_v"):
            assert torch.equal(getattr(big, name), torch.cat([getattr(hg, name) for hg in halves])), f"step {it}: {name}"


# ------------------------------------------------------------------ the training loop -----------------------------------
@pytest.mark.parametrize("mode", ["batched", "per_agent"])
def test_train_loop_learns_with_n_step_returns_from_the_config_alone(mode):
    from dmdqn_b200.train import PRESETS, train_agents
    cfg = dict(PRESETS["shipped_train_py"])
    cfg.update(max_sim_time=600.0, backend="fake", grid_rows=3, grid_cols=3, fake_traci_seed=11, batch_size=16,
               nn_layers=[64, 64], precision="auto", n_step=3)
    history, agents, group = train_agents(cfg, episodes=1, mode=mode, seed=3, learn=True)
    assert group.hp.n_step == 3
    t = len(history)
    assert t > 16 and np.all(group.learn_step.cpu().numpy() == t - 15)      # one learn step per step once 16 are stored
    assert any(h["total_loss"] != 0 for h in history)
    assert np.all(np.isfinite([h["total_loss"] for h in history]))
    assert int(group.debug_views()["tc_error"][0]) == 0
    if mode == "batched":                              # the last step's targets bootstrap up to three steps ahead
        dbg = group.debug_views()
        g = 0.99
        assert np.any(dbg["discount"].cpu().numpy() == np.float32(g * g * g))
        assert torch.any(dbg["next_rows"] != dbg["rows"])
