"""Implicit quantile networks (IQN) on the GPU: the device fractions, the learn step, act and the host API against
tests/iqn_oracle.py, and the bit-equality invariants of the other learn paths."""
import ctypes as C

import numpy as np
import pytest
import torch

import iqn_oracle as IO
import replay_oracle as O
from oracle.dqn import adam_scalars, adam_update_
from parity_util import RTOL, check_nstep_against_oracle, close, copy_state, draw_words, fill_rings, host_ring
from test_gpu_dist import fill, load

pytestmark = pytest.mark.gpu

STATE = ("theta", "theta_tgt", "adam_m", "adam_v", "learn_step", "metrics")


def iqn_group(n, cap, b, h=64, a=4, taus=(8, 8, 32), n_cos=64, kappa=1.0, seed=0, **extra):
    from dmdqn_b200.group import AgentGroup
    cfg = {"nn_layers": [h, h], "replay_buffer_size": cap, "batch_size": b, "learning_rate": 5e-4, "gamma": 0.99,
           "target_update_frequency": 3, "iqn": True, "iqn_num_tau": taus[0], "iqn_num_tau_prime": taus[1],
           "iqn_num_policy_tau": taus[2], "iqn_embedding_dim": n_cos, "quantile_kappa": kappa}
    cfg.update(extra)
    return AgentGroup(n, cfg, action_size=a, seed=seed)


def oracle_for(grp, n, h, a, taus, n_cos, kappa, seed=50, **kw):
    stk = IO.IqnOracle(n, 89, h, a, n_cos=n_cos, n_tau=taus[0], n_tau_prime=taus[1], n_policy=taus[2], kappa=kappa,
                       gamma=0.99, learning_rate=5e-4, target_update_frequency=3, seed0=seed, **kw)
    rng = np.random.default_rng(seed + h + n_cos)
    for k in (1, 3, 5, 7):
        stk.online[k] += torch.as_tensor(rng.standard_normal(stk.online[k].shape).astype(np.float32)) * 0.05
        stk.target[k].copy_(stk.online[k])
    return stk


def backward64(params, states, tau, actions, grad, dh1, dh2, dphi):
    """float64 parameter gradients of one step from the device's own quantile gradient ``grad`` [G, B, N] and ReLU branches:
    relu'(h1), relu'(phi) and relu'(h2) are where the device's dh1 [G, B, H], dphi and dh2 [G, N, B, H] are non-zero (the
    choice of branch at a pre-activation within round-off of 0 becomes an input, as in parity_util.branch_gradients).
    Asserts every mask agrees with the sign of the float64 pre-activation away from kinks."""
    w1, b1, w2, b2, w3, b3, wp, bp = (np.asarray(p, np.float64) for p in params)
    x = np.asarray(states, np.float64)
    c = IO.cos_features(tau, wp.shape[1]).astype(np.float64)                  # [G, B, N, C], the device's rounded features
    z1 = np.einsum("gbd,gdh->gbh", x, w1) + b1[:, None]
    h1 = np.maximum(z1, 0)
    zp = np.einsum("gbnc,gch->gbnh", c, wp) + bp[:, None, None]
    phi = np.maximum(zp, 0)
    z = h1[:, :, None] * phi
    z2 = np.einsum("gbnh,ghk->gbnk", z, w2) + b2[:, None, None]
    h2 = np.maximum(z2, 0)
    m1 = np.asarray(dh1) != 0
    m2 = np.moveaxis(np.asarray(dh2), 1, 2) != 0                               # -> [G, B, N, H]
    mp = np.moveaxis(np.asarray(dphi), 1, 2) != 0
    for pre, m, name in ((z1, m1, "h1"), (zp, mp, "phi"), (z2, m2, "h2")):
        kink = np.abs(pre) < 4 * RTOL * np.abs(pre).max()
        assert not (m & (pre <= 0) & ~kink).any(), f"relu'({name}) set where the pre-activation is clearly negative"
    dZ = np.zeros(h2.shape[:3] + (w3.shape[2],))
    np.put_along_axis(dZ, np.asarray(actions, np.int64)[..., None, None], np.asarray(grad, np.float64)[..., None], 3)
    dh2_ = np.einsum("gbna,gha->gbnh", dZ, w3) * m2
    dz = np.einsum("gbnk,ghk->gbnh", dh2_, w2)
    dphi_ = dz * h1[:, :, None] * mp
    dh1_ = (dz * phi).sum(2) * m1
    return [np.einsum("gbd,gbh->gdh", x, dh1_), dh1_.sum(1), np.einsum("gbnh,gbnk->ghk", z, dh2_), dh2_.sum((1, 2)),
            np.einsum("gbnh,gbna->gha", h2, dZ), dZ.sum((1, 2)), np.einsum("gbnc,gbnh->gch", c, dphi_), dphi_.sum((1, 2))]


def device_fractions(grp, step):
    """The restatement of the fractions the last learn step drew: set 0 [G, B, N] and set 1 [G, B, N']."""
    keys = [int(k) & ((1 << 64) - 1) for k in grp.key.cpu().tolist()]
    rows = grp.iqn_row_base + np.arange(grp.batch_size)
    c = grp.config
    return (np.stack([IO.fractions(k, rows, c["iqn_num_tau"], step, 0) for k in keys]),
            np.stack([IO.fractions(k, rows, c["iqn_num_tau_prime"], step, 1) for k in keys]))


def one_step_against_the_oracle(h, a, taus=(8, 8, 32), n_cos=64, kappa=1.0, steps=1, b=64, clip=None, **extra):
    n, cap = 3, 200
    grp = iqn_group(n, cap, b, h=h, a=a, taus=taus, n_cos=n_cos, kappa=kappa, global_clipnorm=clip, **extra)
    double_dqn = extra.get("double_dqn", True)
    stk = oracle_for(grp, n, h, a, taus, n_cos, kappa, double_dqn=double_dqn)
    load(grp, stk)
    fill(grp, [cap + 40, 150, cap], seed=h + n_cos)
    ring = host_ring(grp)
    obs, nobs, act = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    rng = np.random.default_rng(h + a + n_cos)
    prioritized, n_step = grp.prioritized, grp.n_step
    checked = 0
    for step in range(steps):
        th0 = [torch.stack(x) for x in zip(*[grp.get_weights(i, "online") for i in range(n)])]
        m0 = [torch.stack(x) for x in zip(*[grp.get_weights(i, "m") for i in range(n)])]
        v0 = [torch.stack(x) for x in zip(*[grp.get_weights(i, "v") for i in range(n)])]
        tg0 = grp.theta_tgt.clone()
        for p, q in zip(stk.online, th0):
            p.copy_(q)
        for p, q in zip(stk.target, [torch.stack(x) for x in zip(*[grp.get_weights(i, "target") for i in range(n)])]):
            p.copy_(q)
        if prioritized:
            pr0 = grp.priority.cpu().numpy()
        t_step = int(grp.learn_step_host[0])
        metrics = grp.learn(draw_words(rng, n, b)).cpu().numpy()
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        gblk = grp.grads.clone()
        tau, tau_p = device_fractions(grp, t_step)
        assert np.array_equal(dbg["tau"], tau) and np.array_equal(dbg["tau_prime"], tau_p), "fractions"
        slots, nslots = dbg["rows"] % cap, dbg["next_rows"] % cap
        outs = check_nstep_against_oracle(grp, ring, dbg, n_step, what=f"step {step}")
        take = lambda arr, s: np.stack([arr[g, s[g]] for g in range(n)])
        S, A_, S2 = take(obs, slots), take(act, slots), take(nobs, nslots)
        Rn, disc = (np.stack([o[k] for o in outs]) for k in ("r_hat", "discount"))
        isw = dbg["is_weights"] if prioritized else None
        out = stk.learn_on_batch(S, A_, Rn, S2, disc, tau, tau_p, is_weights=isw, apply=False)
        for key in ("q_all", "q_next", "tq_all"):
            close(dbg[key][..., :a], out[key], what=f"step {step} {key}")
            assert not np.any(dbg[key][..., a:] != 0)
        sel = np.sort(out["q_next"], axis=2)
        tie = (sel[..., -1] - sel[..., -2]) < 4 * RTOL * np.abs(sel).max() if a > 1 else np.zeros(sel.shape[:2], bool)
        assert tie.mean() < 0.1
        close(dbg["target"][~tie], out["T"][~tie], what=f"step {step} target samples")
        close(dbg["theta"], out["theta"], what=f"step {step} theta")
        close(dbg["grad"][~tie], out["grad"][~tie], what=f"step {step} quantile gradient")
        qa = out["q_all"].astype(np.float64).reshape(n, -1)
        hist = np.stack([np.bincount(A_[g], minlength=4) for g in range(n)])
        close(metrics[:, 1], qa.mean(1), scale=np.abs(qa).max(), what="q mean")
        close(metrics[:, 2], qa.std(1), scale=np.abs(qa).max(), rtol=1e-4, what="q std")
        assert np.array_equal(metrics[:, 3:7], hist) and np.all(metrics[:, 7] == 1)
        if prioritized:
            pr1 = grp.priority.cpu().numpy()
            for g in range(n):
                if tie[g].any():
                    continue
                last = {s_: r for r, s_ in enumerate(slots[g])}      # a slot drawn twice keeps its last row's priority
                rows_ = np.array([last[s_] for s_ in slots[g]])
                close(pr1[g, slots[g]], O.priority_of(out["row_loss"][g][rows_], 0.6, 1e-6),
                      what=f"step {step} net {g}: priorities")
                untouched = np.ones(cap, bool); untouched[slots[g]] = False
                assert np.array_equal(pr1[g, untouched], pr0[g, untouched])
        g64 = backward64([p.numpy() for p in th0], S, tau, A_, dbg["grad"], dbg["dh1"], dbg["dh2_pass"], dbg["dphi_pass"])
        alpha_t, eps_t = adam_scalars(int(grp.learn_step_host[0]), 5e-4, "keras")
        L = grp.layout
        for i in range(n):
            if tie[i].any():
                continue
            checked += 1
            close(metrics[i, 0], out["loss"][i], what=f"step {step} net {i} loss")
            got = grp.unpack(gblk[i])
            for k in range(8):
                close(got[k].numpy(), g64[k][i], what=f"step {step} net {i} grad[{k}]")
            g_all = [x.clone() for x in got]
            if clip is not None:
                nrm = float(np.sqrt(sum(float((x.double() ** 2).sum()) for x in g_all)))
                close(grp.grad_norms.cpu().numpy()[i], nrm, what="norm")
                s = np.float32(clip / max(nrm, clip))
                if s != 1:
                    g_all = [x * s for x in g_all]
            th, mm, vv = grp.get_weights(i, "online"), grp.get_weights(i, "m"), grp.get_weights(i, "v")
            for k in range(8):
                p, m_, v_ = th0[k][i].clone(), m0[k][i].clone(), v0[k][i].clone()
                adam_update_(p, g_all[k], m_, v_, alpha_t, eps_t)
                close(th[k].numpy(), p.numpy(), what=f"step {step} net {i} theta[{k}]")
                close(mm[k].numpy(), m_.numpy(), what=f"step {step} net {i} m[{k}]")
                close(vv[k].numpy(), v_.numpy(), rtol=2 * RTOL, what=f"step {step} net {i} v[{k}]")
        W3 = gblk[:, L.w3:L.w3 + grp.hidden * 4].view(n, grp.hidden, 4)
        assert not torch.any(W3[:, :, a:] != 0) and not torch.any(gblk[:, L.b3 + a:L.b3 + 4] != 0)
        ls = int(grp.learn_step_host[0])
        if extra.get("tau") is not None:
            tau_s = float(np.float32(extra["tau"]))
            close(grp.theta_tgt.cpu().numpy(), (tau_s * grp.theta + (1.0 - tau_s) * tg0).cpu().numpy(), what="polyak")
        elif ls % 3 == 0:
            assert torch.equal(grp.theta_tgt, grp.theta)
        else:
            assert torch.equal(grp.theta_tgt, tg0)
    assert checked > 0
    return grp


@pytest.mark.parametrize("h,a,taus,n_cos,kappa", [(64, 2, (1, 1, 1), 4, 1.0), (64, 4, (8, 8, 32), 64, 1.0),
                                                  (128, 3, (13, 5, 7), 128, 0.0), (256, 4, (8, 8, 32), 64, 1.0),
                                                  (256, 2, (64, 64, 64), 64, 1.0), (512, 4, (13, 5, 7), 64, 0.0),
                                                  (512, 3, (8, 8, 32), 4, 1.0)])
def test_one_step_matches_the_oracle(h, a, taus, n_cos, kappa):
    one_step_against_the_oracle(h, a, taus, n_cos, kappa)


@pytest.mark.parametrize("extra", [{"sample_mode": "prioritized"}, {"n_step": 3}, {"double_dqn": False}, {"tau": 0.05},
                                   {"clip": 0.05}, {"clip": 1e6}])
def test_learn_variants_match_the_oracle(extra):
    one_step_against_the_oracle(128, 4, steps=3, **extra)


def test_thirty_consecutive_steps_each_against_the_oracle():
    """30 steps, the oracle's state reset to the device's before each (so every step checks the kernels)."""
    one_step_against_the_oracle(64, 4, (8, 6, 16), 16, steps=30, b=32)


def test_free_running_trajectory_follows_the_oracle():
    """30 steps with the oracle on its own weights, Adam state and target sync from the same start: the device's sampled
    rows and fractions (both checked bit for bit elsewhere) feed the oracle; the losses and the final online and target
    weights agree to 1e-4 of their magnitude (30 steps of float32 rounding, compounded through Adam)."""
    n, cap, b, h, a, taus, n_cos = 2, 200, 32, 64, 4, (8, 6, 16), 16
    grp = iqn_group(n, cap, b, h=h, a=a, taus=taus, n_cos=n_cos)
    stk = oracle_for(grp, n, h, a, taus, n_cos, 1.0)
    load(grp, stk)
    fill(grp, cap, seed=17)
    ring = host_ring(grp)
    obs, nobs, act = grp.obs.cpu().numpy()[..., :89], grp.next_obs.cpu().numpy()[..., :89], grp.act_ring.cpu().numpy()
    rng = np.random.default_rng(18)
    take = lambda arr, s: np.stack([arr[g, s[g]] for g in range(n)])
    for step in range(30):
        t_step = int(grp.learn_step_host[0])
        metrics = grp.learn(draw_words(rng, n, b)).cpu().numpy()
        dbg = {k: v.cpu().numpy() for k, v in grp.debug_views().items()}
        tau, tau_p = device_fractions(grp, t_step)
        slots, nslots = dbg["rows"] % cap, dbg["next_rows"] % cap
        outs = check_nstep_against_oracle(grp, ring, dbg, 1, what=f"step {step}")
        Rn, disc = (np.stack([o[k] for o in outs]) for k in ("r_hat", "discount"))
        out = stk.learn_on_batch(take(obs, slots), take(act, slots), Rn, take(nobs, nslots), disc, tau, tau_p)
        close(metrics[:, 0], out["loss"], rtol=1e-4, what=f"step {step} loss")
    for i in range(n):
        for which, ref in (("online", stk.online), ("target", stk.target)):
            for k, w in enumerate(grp.get_weights(i, which)):
                close(w.numpy(), ref[k][i].numpy(), rtol=1e-4, what=f"net {i} {which}[{k}]")


def test_one_group_of_eight_equals_two_groups_of_four_and_a_nonzero_row_base():
    big = iqn_group(8, 200, 64, h=128, seed=4)
    fill(big, 200, seed=5)
    halves = [iqn_group(4, 200, 64, h=128, seed=4 + 4 * k) for k in range(2)]
    for k, hg in enumerate(halves):
        copy_state(hg, big, slice(4 * k, 4 * k + 4))
        hg.key.copy_(big.key[4 * k:4 * k + 4])
    rng = np.random.default_rng(6)
    for it in range(3):
        w = draw_words(rng, 8, 64)
        big.learn(w)
        for k, hg in enumerate(halves):
            hg.learn(w[4 * k:4 * k + 4].contiguous())
        torch.cuda.synchronize()
        for name in STATE:
            assert torch.equal(getattr(big, name), torch.cat([getattr(hg, name) for hg in halves])), f"step {it}: {name}"
    shifted = iqn_group(2, 200, 64, h=64, seed=8)
    fill(shifted, 200, seed=9)
    shifted.iqn_row_base = 64
    t0 = int(shifted.learn_step_host[0])
    shifted.learn(draw_words(rng, 2, 64))
    dbg = shifted.debug_views()
    tau, tau_p = device_fractions(shifted, t0)
    assert np.array_equal(dbg["tau"].cpu().numpy(), tau) and np.array_equal(dbg["tau_prime"].cpu().numpy(), tau_p)


def test_act_matches_the_oracle_skips_exploring_agents_and_acts_on_the_target():
    n, h, a, taus, n_cos = 64, 128, 3, (8, 8, 32), 64
    for hh, kk in ((h, taus), (512, (8, 8, 64)), (64, (8, 8, 1))):
        grp = iqn_group(n, 100, 32, h=hh, a=a, taus=kk, n_cos=n_cos)
        stk = oracle_for(grp, n, hh, a, kk, n_cos, 1.0)
        load(grp, stk)
        rng = np.random.default_rng(3)
        obs = rng.integers(-1, 20, (n, 89)).astype(np.float32) * np.float32(0.125)
        acts, q = grp.act(obs, return_q=True)
        ref_a, ref_q = stk.act(obs, np.zeros(n), np.zeros(n, np.uint32), np.zeros(n, np.uint32))
        q = q.cpu().numpy()
        close(q[:, :a], ref_q, what=f"h {hh}: policy Q")
        assert not np.any(q[:, a:] != 0)
        srt = np.sort(ref_q, 1)
        ok = (srt[:, -1] - srt[:, -2]) > 4 * RTOL * np.abs(ref_q).max()
        assert ok.mean() > 0.9 and np.array_equal(acts.cpu().numpy()[ok], ref_a[ok])
        eps = np.where(np.arange(n) % 2 == 0, 1.0, 0.0)
        acts2, q2 = grp.act(obs, eps=eps, return_q=True)
        q2 = q2.cpu().numpy()
        assert np.all(np.isnan(q2[::2])) and np.array_equal(q2[1::2], q[1::2])
        assert np.all(acts2.cpu().numpy() < a)
    grp.theta_tgt.mul_(0.5)
    _, qt = grp.act(obs, return_q=True, target=True)
    ref = stk.policy_q([p * 0.5 for p in stk.target], obs[:, None])[:, 0]
    close(qt.cpu().numpy()[:, :a], ref, what="target policy Q")


def _twins(n=6, cap=200, b=64, **extra):
    a, c = (iqn_group(n, cap, b, h=128, seed=7, **extra) for _ in range(2))
    for g in (a, c):
        fill(g, cap, seed=8)
    return a, c


@pytest.mark.parametrize("extra", [{}, {"sample_mode": "prioritized"}])
def test_captured_learn_equals_plain_learn(extra):
    a, c = _twins(**extra)
    replay, draws = c.capture_learn()
    a.learn(draws.clone())
    rng = np.random.default_rng(9)
    for it in range(4):
        w = draw_words(rng, 6, 64)
        draws.copy_(w)
        replay()
        a.learn(w)
        torch.cuda.synchronize()
        for name in STATE + (("priority",) if a.prioritized else ()):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name}"


def test_captured_step_host_equals_step_host():
    n, b = 6, 64
    a, c = _twins(n=n, b=b)
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
        assert torch.equal(ma, mc), f"step {it}: metrics"
        for name in STATE + ("obs",):
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name}"


def test_reruns_repeat_and_a_nan_gradient_buffer_changes_nothing():
    a, c = _twins(n=3)
    c.grads.fill_(float("nan"))
    rng = np.random.default_rng(16)
    for it in range(3):
        w = draw_words(rng, 3, 64)
        a.learn(w)
        c.learn(w)
        torch.cuda.synchronize()
        for name in STATE:
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name}"
        end = a.layout.end                            # every float of [0, end) is written
        assert torch.equal(a.grads[:, :end], c.grads[:, :end]), f"step {it}: grads"
        da, dc = a.debug_views(), c.debug_views()
        for key in ("tau", "tau_prime", "target", "theta", "grad", "q_all", "q_next", "tq_all"):
            assert torch.equal(da[key], dc[key]), key


def test_inactive_networks_stay_untouched_with_zero_metrics():
    grp = iqn_group(3, 200, 64, h=64, seed=2)
    fill(grp, [200, 20, 200], seed=3)                  # network 1 holds fewer than batch transitions
    mask = np.array([1, 1, 0], np.uint8)               # network 2 is masked out
    before = {k: getattr(grp, k).clone() for k in ("theta", "theta_tgt", "adam_m", "adam_v")}
    grp.metrics.fill_(7.0)
    metrics = grp.learn(draw_words(np.random.default_rng(1), 3, 64), mask=mask).cpu().numpy()
    assert np.all(metrics[1:] == 0) and metrics[0, 7] == 1
    for k, v in before.items():
        assert torch.equal(getattr(grp, k)[1:], v[1:]), k
        assert not torch.equal(getattr(grp, k)[0], v[0]) or k == "theta_tgt", k


def test_shared_parameters_nccl_path_and_two_simulated_ranks():
    from dmdqn_b200 import _native as N
    from dmdqn_b200.parallel import SharedParameterStep
    a, c = (iqn_group(4, 100, 64, h=128, seed=21, share_parameters=True) for _ in range(2))
    for g in (a, c):
        fill(g, 100, seed=22)
    step = SharedParameterStep.for_group(a, fused=False)
    with pytest.raises(ValueError, match="iqn"):
        SharedParameterStep.for_group(a, fused=True)
    for it in range(3):
        a._gen.manual_seed(100 + it)
        c._gen.manual_seed(100 + it)
        step.step()
        d = c.draw_words((1, c.batch_size))
        N.check(c.lib.dmdqn_learn_grads_iqn(C.byref(c.dims), C.byref(c.hp), C.byref(c.iqn_args), C.byref(c.replay),
                                            C.byref(c.nets), d.data_ptr(), None, 64, c.grads.data_ptr(), c.metrics.data_ptr(),
                                            c.workspace.data_ptr(), c.workspace.numel(), None))
        N.check(c.lib.dmdqn_adam_apply_iqn(C.byref(c.dims), C.byref(c.hp), C.byref(c.nets), c.n_cos, c.grads.data_ptr(), 0.0,
                                           None, c.workspace.data_ptr(), c.workspace.numel(), None))
        torch.cuda.synchronize()
        for name in STATE:
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name}"
    # two ranks of batch B (row_base 0 and B) sum to one process's gradient of batch 2B over the same rows
    # (draws with replacement and raw rewards: a row depends on its own word only)
    kw = dict(h=64, seed=30, share_parameters=True, sample_mode="replacement", normalize_rewards=False)
    one = iqn_group(4, 100, 128, **kw)
    ranks = [iqn_group(4, 100, 64, **kw) for _ in range(2)]
    for g in [one] + ranks:
        fill(g, 100, seed=31)
    idx = draw_words(np.random.default_rng(32), 1, 128)
    one._grads_call(one.hp, idx.data_ptr(), None, 128, one.grads.data_ptr(), one._stream)
    total = torch.zeros_like(one.grads)
    for r, g in enumerate(ranks):
        g.iqn_row_base = 64 * r
        part = idx[:, 64 * r:64 * r + 64].contiguous()
        g._grads_call(g.hp, part.data_ptr(), None, 128, g.grads.data_ptr(), g._stream)
        total += g.grads
    torch.cuda.synchronize()
    for k, (x, y) in enumerate(zip(one.unpack(total[0]), one.unpack(one.grads[0]))):
        close(x.numpy(), y.numpy(), what=f"two ranks grad[{k}]")


def test_weights_round_trip_and_initial_trunk_equals_a_plain_group(tmp_path):
    from dmdqn_b200.agent import DQNAgent
    from dmdqn_b200.group import AgentGroup
    grp = iqn_group(2, 100, 32, h=64, a=3, n_cos=16)
    ws = grp.get_weights(1)
    assert [tuple(w.shape) for w in ws] == [(89, 64), (64,), (64, 64), (64,), (64, 3), (3,), (16, 64), (64,)]
    new = [w + 0.25 for w in ws]
    grp.set_weights(0, new, sync_target=True)
    for x, y in zip(grp.get_weights(0), new):
        assert torch.equal(x, y)
    assert torch.equal(grp.theta[0], grp.theta_tgt[0])
    cfg = {"nn_layers": [64, 64], "replay_buffer_size": 100, "batch_size": 32, "iqn": True, "iqn_embedding_dim": 16}
    ag = DQNAgent(89, 3, "a0", cfg)
    ag._g.set_weights(0, new)
    path = str(tmp_path / "m.pt")
    ag.save_model(path)
    other = DQNAgent(89, 3, "a1", cfg)
    assert other.load_model(path)
    for x, y in zip(other._g.get_weights(0), new):
        assert torch.equal(x, y)
    base = {"nn_layers": [64, 64], "replay_buffer_size": 100, "batch_size": 32, "precision": "fp32"}
    q = AgentGroup(3, dict(base, iqn=True), seed=5)
    p = AgentGroup(3, dict(base), seed=5)
    for g in range(3):
        for x, y in zip(q.get_weights(g)[:6], p.get_weights(g)):
            assert torch.equal(x, y)


def test_iqn_false_is_bit_identical_to_a_group_without_the_key():
    from dmdqn_b200.group import AgentGroup
    base = {"nn_layers": [128, 128], "replay_buffer_size": 200, "batch_size": 64, "target_update_frequency": 3}
    a = AgentGroup(4, dict(base), seed=3)
    c = AgentGroup(4, dict(base, iqn=False, iqn_num_tau=3, iqn_embedding_dim=8), seed=3)
    for g in (a, c):
        fill_rings(g, 200, seed=4)
    rng = np.random.default_rng(5)
    for it in range(3):
        w = draw_words(rng, 4, 64)
        a.learn(w)
        c.learn(w)
        torch.cuda.synchronize()
        for name in STATE:
            assert torch.equal(getattr(a, name), getattr(c, name)), f"step {it}: {name}"
    assert a.layout.stride == c.layout.stride


def test_train_loop_runs_iqn_from_the_config():
    from dmdqn_b200.train import PRESETS, train_agents
    cfg = dict(PRESETS["shipped_train_py"])
    cfg.update(max_sim_time=600.0, backend="fake", grid_rows=3, grid_cols=3, fake_traci_seed=11, batch_size=16,
               nn_layers=[64, 64], precision="auto", iqn=True, sample_mode="prioritized", n_step=3)
    history, agents, group = train_agents(cfg, episodes=1, mode="batched", seed=3, learn=True)
    t = len(history)
    assert group.iqn and group.hp.precision == 0
    assert t > 16 and np.all(group.learn_step.cpu().numpy() == t - 15)
    losses = [h["total_loss"] for h in history]
    assert np.all(np.isfinite(losses)) and any(x != 0 for x in losses)
